// vargeno_main.cpp -- `vargeno-b200`: the reference's command line (src/qv.cc:1853-1881, 2109-2131) in front of the
// B200 hot path.  `geno` is the drop-in for the hot path; `index` writes the same five files as the reference's
// `vargeno index` (byte-identical), with the sort / collapse / Bloom-filter work done on the GPU.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "geno_host.h"

static void print_help()
{
	fprintf(stderr, "Usage: vargeno-b200 <option> [option parameters ...]\n");
	fprintf(stderr, "Option  Description                   Parameters\n");
	fprintf(stderr, "------  -----------                   ----------\n");
	fprintf(stderr, "geno    Perform genotyping (B200)     <index_prefix> <input FASTQ> <input SNPs in VCF> <output file in VCF> "
	                "[--gpus N] [--chunk-mb M] [--verbose]\n");
	fprintf(stderr, "        (<input FASTQ>: one file or a comma-separated list read back to back; each plain or gzip; or BAM files only)\n");
	fprintf(stderr, "        (gzip input is inflated on the GPU: BGZF over all GPUs, single-stream gzip on the first GPU only;\n"
	                "         pipes and lists that mix plain and gzip files are inflated on the host)\n");
	fprintf(stderr, "        (the VCF is written on the GPU; an output name ending in .gz gets BGZF, as bgzip writes it)\n");
	fprintf(stderr, "        (BAM, unaligned or aligned: the reads `samtools fastq` gives, inflated and converted on the GPU; each file\n"
	                "         on one GPU, largest first; a list may not mix BAM and other files; VGB_HOST_INFLATE and\n"
	                "         VGB_SEQUENTIAL_READER do not apply)\n");
	fprintf(stderr, "geno-samples  Genotype a cohort (B200)  <index_prefix> <samples.tsv> <input SNPs in VCF> <output dir> "
	                "[--gpus N] [--chunk-mb M] [--bgzf] [--verbose]\n");
	fprintf(stderr, "        (samples.tsv: one sample per line, <name><TAB><reads>, reads as for geno; names of [A-Za-z0-9._-], unique;\n"
	                "         '#' lines and blank lines skipped.  Writes <output dir>/<name>.vcf (--bgzf: <name>.vcf.gz), the file geno writes for that sample.\n"
	                "         The index is loaded once per GPU and each GPU takes whole samples, largest first: a sample never\n"
	                "         spans GPUs, so a cohort smaller than --gpus leaves GPUs idle.  A sample whose input fails gets no VCF\n"
	                "         and the exit status is 1; the other samples go on)\n");
	fprintf(stderr, "filt    Keep the reference-dictionary entries near SNPs   <ref.dict> <snp_locs> <out.dict>   (the reference's hidden `filt`)\n");
	fprintf(stderr, "index   Build the index (B200)         <input FASTA> <input SNPs in VCF> <index_prefix> [--gpu D] [--no-lite] [--verbose]\n");
	fprintf(stderr, "        (the same files as the reference's `vargeno index`, byte for byte; --no-lite skips the 2.3 GB .ref.bf.lite.bf that nothing reads)\n");
}

int main(int argc, const char *argv[])
{
	if (argc < 2) { print_help(); return 0; }
	const std::string opt = argv[1];
	if (opt == "geno" || opt == "geno-samples") {
		std::string pos[4];
		int npos = 0, gpus = 1;
		uint64_t chunk_mb = 256;
		bool verbose = false, bgzf = false;
		for (int i = 2; i < argc; i++) {
			if (!strcmp(argv[i], "--gpus") && i + 1 < argc) gpus = atoi(argv[++i]);
			else if (!strcmp(argv[i], "--chunk-mb") && i + 1 < argc) chunk_mb = strtoull(argv[++i], nullptr, 10);
			else if (!strcmp(argv[i], "--verbose")) verbose = true;
			else if (!strcmp(argv[i], "--bgzf") && opt == "geno-samples") bgzf = true;
			else if (npos < 4) pos[npos++] = argv[i];
			else npos++;
		}
		if (npos != 4 || gpus < 1 || chunk_mb < 1 || chunk_mb > 4000) { print_help(); return EXIT_FAILURE; }   // arg_check, src/qv.cc:1875-1881
		if (opt == "geno-samples") return vgh::run_geno_samples(pos[0], pos[1], pos[2], pos[3], gpus, chunk_mb << 20, verbose, bgzf);
		return vgh::run_geno(pos[0], pos[1], pos[2], pos[3], gpus, chunk_mb << 20, verbose);
	}
	if (opt == "index") {
		std::string pos[3], dump, locs;
		int npos = 0, dev = 0;
		bool verbose = false, lite = true;
		for (int i = 2; i < argc; i++) {
			if (!strcmp(argv[i], "--gpu") && i + 1 < argc) dev = atoi(argv[++i]);
			else if (!strcmp(argv[i], "--no-lite")) lite = false;
			else if (!strcmp(argv[i], "--snp-locs") && i + 1 < argc) locs = argv[++i];
			else if (!strcmp(argv[i], "--dump-parse") && i + 1 < argc) dump = argv[++i];
			else if (!strcmp(argv[i], "--verbose")) verbose = true;
			else if (npos < 3) pos[npos++] = argv[i];
			else npos++;
		}
		if (npos != 3 || dev < 0) { print_help(); return EXIT_FAILURE; }   // arg_check, src/qv.cc:1875-1881
		return vgh::run_index(pos[0], pos[1], pos[2], dev, verbose, dump, lite, locs);
	}
	if (opt == "filt") {              // dict_filt (src/qv.cc:2009-2025): <ref.dict> <snp_locs> <out.dict>
		if (argc != 5) { print_help(); return EXIT_FAILURE; }
		return vgh::run_filt(argv[2], argv[3], argv[4]);
	}
	if (opt == "fastq-chunks") {      // host-logic check, no GPU: how the FASTQ input would be cut into record-aligned chunks
		std::string files;
		uint64_t bytes = 256ull << 20;
		bool timing = false;
		int parallel = 0;
		for (int i = 2; i < argc; i++) {
			if (!strcmp(argv[i], "--time")) timing = true;
			else if (!strcmp(argv[i], "--parallel") && i + 1 < argc) parallel = atoi(argv[++i]);
			else if (!strcmp(argv[i], "--chunk-bytes") && i + 1 < argc) bytes = strtoull(argv[++i], nullptr, 10);
			else if (!strcmp(argv[i], "--chunk-mb") && i + 1 < argc) bytes = strtoull(argv[++i], nullptr, 10) << 20;
			else files = argv[i];
		}
		if (files.empty() || bytes < 16) { print_help(); return EXIT_FAILURE; }
		return vgh::run_fastq_chunks(files, bytes, timing, parallel);
	}
	if (opt == "vcf-rewrite") {       // host-logic check, no GPU: chrlens mapping + GQ + VCF rewrite from a table of calls
		if (argc != 6) { print_help(); return EXIT_FAILURE; }
		return vgh::run_vcf_rewrite(argv[2], argv[3], argv[4], argv[5]);
	}
	if (opt == "help") { print_help(); return EXIT_SUCCESS; }
	print_help();
	return EXIT_FAILURE;
}
