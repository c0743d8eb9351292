/*
 * vgb200.h -- C ABI of the B200-native `vargeno geno` hot path (libvgb200.so).
 *
 * The reference has no plugin / FFI interface: its boundary is the process
 * (`vargeno geno <prefix> <reads.fq> <snps.vcf> <out.vcf>`, /root/reference/src/qv.cc:2109-2207) and,
 * inside it, one function: static void genotype(FILE*, FILE*, FILE*, FILE*, string, string)
 * (src/qv.cc:475) plus the globals ref_bf / snp_bf (src/qv.cc:38-39).  This header is the seam a
 * maintainer would cut through that function (INTEGRATION.md shows the patch): each entry point
 * below names the reference lines it replaces.
 *
 * Conventions: plain C types only, 0 = ok, negative = error (vgb_last_error() has the text), no
 * exceptions, no global state.  One context per GPU; a context is driven by one host thread at a
 * time; CUDA streams and events are internal.  All host buffers stay owned by the caller; the
 * library copies what it needs before the call returns unless stated otherwise.
 *
 * There is NO CPU fallback: every compute entry point fails with VGB_E_CUDA when no sm_100-class
 * device is usable.
 */
#ifndef VGB200_H
#define VGB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VGB_ABI_VERSION 2

typedef struct vgb_ctx vgb_ctx;

enum {
	VGB_OK          = 0,
	VGB_E_ARG       = -1,   /* bad argument / call order */
	VGB_E_CUDA      = -2,   /* CUDA runtime error or no usable device */
	VGB_E_FORMAT    = -3,   /* FASTQ chunk violates the input contract (see vgb_submit_fastq) */
	VGB_E_INDEX     = -4,   /* index image violates the format contract */
	VGB_E_NCCL      = -5,
	VGB_E_OVERFLOW  = -6    /* a read produced more hit contexts than the reference's arrays hold (2000, qv.cc:709) */
};

enum {
	VGB_CFG_TRACE = 1u << 0  /* keep a per-read vote record (vgb_fetch_read_results); costs 24 B/read */
};

typedef struct {
	int32_t  device;            /* CUDA device ordinal */
	int32_t  world_size;        /* >= 1; > 1 enables vgb_allreduce_pileup over NCCL */
	int32_t  rank;
	uint32_t flags;             /* VGB_CFG_* */
	const void *nccl_unique_id; /* 128-byte ncclUniqueId shared by all ranks (rank 0 gets one from vgb_nccl_unique_id); NULL if world_size == 1 */
	uint64_t max_chunk_bytes;   /* largest FASTQ chunk that will be submitted; 0 = 256 MiB */
} vgb_config;

/* The index as the reference's files hold it (SURVEY.md 3.3 table; written by src/dictgen.c:63-275 and
 * src/generate_bf.h:83-89).  Record arrays are the raw little-endian on-disk records, still sorted by k-mer:
 * entry RANK matters (the reference's block scan is rank-strided, src/qv.cc:355-363,444-452). */
typedef struct {
	const uint8_t  *ref_records;  uint64_t n_ref;       /* n_ref     x 13 B {u64 kmer, u32 pos, u8 flag} */
	const uint32_t *ref_aux;      uint64_t n_ref_aux;   /* n_ref_aux x 10 u32 */
	const uint8_t  *snp_records;  uint64_t n_snp;       /* n_snp     x 16 B {u64 kmer, u32 pos, u8 snp, u8 flag, u8 rf, u8 af} */
	const uint8_t  *snp_aux;      uint64_t n_snp_aux;   /* n_snp_aux x 78 B {u64 kmer, 10 x {u32 pos, u8 snp, u8 rf, u8 af}} */
	const uint64_t *ref_bf_words; uint64_t ref_bf_bits; uint64_t ref_bf_nwords;  /* sdsl bit_vector payload; nwords may cover only the addressable prefix */
	const uint64_t *snp_bf_words; uint64_t snp_bf_bits; uint64_t snp_bf_nwords;
} vgb_index_view;

/* result of one dictionary probe (vgb_lookup_kmers) */
typedef struct {
	uint32_t ref_pos;      /* kmer_entry.pos (aux row index if ref_flag == 1) */
	uint32_t snp_pos;
	uint32_t ref_block_lo; /* ref_jumpgate[HI32]            (src/qv.cc:219) */
	uint32_t ref_block_n;  /* check_block_size()            (src/qv.cc:242-264) */
	uint32_t snp_block_lo; /* snp_jumpgate[HI24]            (src/qv.cc:394) */
	uint32_t snp_block_n;
	uint8_t  ref_found, ref_flag;
	uint8_t  snp_found, snp_flag, snp_info;
	uint8_t  ref_bf, snp_bf; /* BloomFilter::check_value(LO32) / (LO40), src/qv.cc:955-956 */
	uint8_t  pad;
} vgb_hit;

/* per-read vote record; same layout as the oracle's vgo_read_result */
typedef struct {
	uint32_t flags;      /* VGB_RF_* */
	uint32_t target;     /* winning read position (valid when VGB_RF_PROCESS) */
	uint16_t freq;       /* votes of the best position */
	uint16_t n_ref;      /* hit contexts recorded from the reference dictionary in the final pass */
	uint16_t n_snp;      /* ... from the SNP dictionary */
	uint16_t passes;     /* 0 skipped, 1 forward only, 2 forward + reverse complement */
	uint64_t ctx_hash;   /* order-independent digest of all hit contexts of the final pass */
} vgb_read_result;

enum {
	VGB_RF_SKIPPED = 1u << 0, VGB_RF_REVCOMPL = 1u << 1, VGB_RF_PROCESS = 1u << 2,
	VGB_RF_AMBIGUOUS = 1u << 3, VGB_RF_HASBEST = 1u << 4
};

typedef struct {
	uint64_t reads, skipped_n, passes, placed;
	uint64_t exact_lookups;      /* dictionary queries on the reads' own k-mers (2 per k-mer per pass) */
	uint64_t nbr_query_lookups;  /* dictionary queries on substituted k-mers */
	uint64_t nbr_scan_reads;     /* strided entry reads of the small-block scan */
	uint64_t bf_probes;
	uint64_t lowq_kmers;
	uint64_t events;             /* hit contexts recorded, all passes */
	uint64_t pileup_incr;        /* counter increments */
	uint64_t big_kmers;
	uint64_t bad_records;        /* records violating the input contract (first error code in vgb_sync) */
	uint64_t chunks, chunk_bytes;
	double   gpu_ms_parse, gpu_ms_geno;   /* CUDA-event time of the K1 kernels (BGZF chunks: the inflate kernel included) and of the per-read
	                                        * kernels.  The hand-over kernels of a chunk run on a second stream under the next chunk's
	                                        * kernels, so these are sums of intervals that overlap; with VGB_NO_TAIL_OVERLAP set in the
	                                        * environment (read at vgb_index_upload) every kernel runs alone and the sums are durations */
	uint64_t kernel_launches;
	uint64_t freq_wrap_reads;    /* reads with more than 255 votes for one position: the reference's uint8 counter wraps there
	                                (src/qv.cc:57-93); never silently used -- vgb_sync fails with VGB_E_OVERFLOW */
} vgb_stats;

/* ---- life cycle ---- */
int  vgb_abi_version(void);
int  vgb_ctx_create(vgb_ctx **out, const vgb_config *cfg);
void vgb_ctx_destroy(vgb_ctx *ctx);
const char *vgb_last_error(const vgb_ctx *ctx);   /* ctx may be NULL: error of the last failed vgb_ctx_create */
int  vgb_nccl_unique_id(void *out128);            /* ncclGetUniqueId through the dlopen'ed libnccl */
/* Joins a context that was created with world_size == 1 to a communicator afterwards (collective: every rank calls it).
 * Lets a host create and load all of its contexts first and start the collective NCCL initialisation only when every
 * rank got that far -- a rank that fails early can then not leave the others blocked in ncclCommInitRank. */
int  vgb_comm_init(vgb_ctx *ctx, int32_t world_size, int32_t rank, const void *nccl_unique_id);

/* ---- index: replaces the dictionary / jumpgate / pileup construction of src/qv.cc:519-695 and the
 *      Bloom filter loads of src/qv.cc:2140-2144 ---- */
int  vgb_index_upload(vgb_ctx *ctx, const vgb_index_view *view);
int  vgb_site_count(vgb_ctx *ctx, uint64_t *n_sites);   /* positions with ref != 0 || alt != 0 in the static pileup */
/* per site, position order: 1-based concatenated position, ref | alt << 2, ref_freq, alt_freq (src/qv.cc:655-658) */
int  vgb_fetch_sites(vgb_ctx *ctx, uint32_t *pos, uint8_t *code, uint8_t *ref_freq, uint8_t *alt_freq, uint64_t n_sites);

/* ---- reads: replaces the FASTQ loop src/qv.cc:760-1558 ----
 * chunk = FASTQ text that starts at a record boundary and holds complete 4-line records only.  Contract
 * (what the reference needs to behave, SURVEY.md 3.3): lines <= 1022 characters, no blank lines, bases in
 * ACGTNacgtn within the first 32*floor(len/32) characters, quality line at least floor(len/32) long.
 * Violations are counted and reported by vgb_sync as VGB_E_FORMAT; such records contribute nothing.
 * Asynchronous: returns once the chunk is staged; host memory may be reused when the call returns.
 * Buffers obtained from vgb_pinned_buffer are copied without an extra staging pass. */
int  vgb_pinned_buffer(vgb_ctx *ctx, int slot, char **ptr, uint64_t *capacity);   /* slot 0 or 1; waits until the slot is free */
int  vgb_submit_fastq(vgb_ctx *ctx, const char *chunk, uint64_t nbytes, uint64_t first_read_id);
int  vgb_submit_fastq_device(vgb_ctx *ctx, const char *device_chunk, uint64_t nbytes, uint64_t first_read_id);
/* BGZF input (blocked gzip, as bgzip / htslib write it): the gzip members of a chunk go over PCIe compressed and are inflated
 * on the device, one warp per member.  `comp` holds the members back to back (host memory; a vgb_pinned_buffer is copied without
 * staging), members[i] locates the raw DEFLATE payload of member i inside it and gives its ISIZE.  A chunk is a run of whole
 * members, so it may begin and end inside a record: the caller puts the last members of the previous chunk (at least 8 KiB of
 * text, or everything back to the start of the input) in front again and passes their inflated size as overlap_bytes -- the
 * chunk then processes exactly the records that end behind that point.  last_chunk: the input ends with this chunk (a trailing
 * partial record is a format error instead of the next chunk's business).  CRC32 of the members is not verified; a member that
 * does not inflate to its ISIZE is reported by vgb_sync as VGB_E_FORMAT. */
typedef struct { uint32_t comp_offset, comp_len, out_len; } vgb_bgzf_member;
int  vgb_submit_bgzf(vgb_ctx *ctx, const void *comp, uint64_t comp_bytes, const vgb_bgzf_member *members, uint32_t n_members,
                     uint64_t overlap_bytes, int last_chunk);
/* Single-stream gzip input (gzip, pigz, Python's gzip: one member or several back to back, no BGZF index): inflated on the device.
 * The caller feeds a stream's bytes in order, in pieces of any size up to max_chunk_bytes (host memory; a vgb_pinned_buffer is
 * copied without staging; the buffer may be reused when the call returns).  first: a new gzip stream starts with this piece (the
 * last 32 KiB of text of the previous stream stay in front of it, so a record may span two streams, as two files read back to
 * back); last: the input ends with this piece (a trailing partial record is a format error).  The caller never needs to know block
 * boundaries or the compression ratio: the library keeps the exact bit cursor, the compressed bytes not consumed yet and the last
 * 32 KiB of text on the device.  Bytes behind the last member that do not start a gzip member end the input.  A corrupt or
 * truncated stream, a member whose CRC32 or ISIZE does not match its text, and a single DEFLATE block that needs more than
 * max_chunk_bytes of input or of text are reported by vgb_sync as VGB_E_FORMAT.  One context inflates a stream. */
int  vgb_submit_gzip(vgb_ctx *ctx, const void *comp, uint64_t comp_bytes, int first, int last);
/* BAM input (unaligned or aligned BAM): the reads are the FASTQ records `samtools fastq` writes with its default settings, in file
 * order -- secondary and supplementary records (flag 0x900) and records without bases are skipped, a record with flag 0x10 is
 * turned back to the sequenced orientation, bases are =ACMGRSVTWYHKDBN (IUPAC codes other than N stay format errors), quality is
 * qual + 33, or 1 for a record stored without quality.  A call takes whole BGZF members of one BAM file, in file order (as for
 * vgb_submit_bgzf: `comp` holds them back to back, members[i] locates the DEFLATE payload of member i and gives its ISIZE), with
 * an ISIZE sum of at most max_chunk_bytes; max_chunk_bytes must be at most 1 GiB.  first: a new file starts with this call (its
 * header comes first); last: the file ends with it.  A context takes several files one after the other.  The members are inflated
 * and the records framed and converted on the device; the bytes a call does not consume (a header not complete yet, the record cut
 * by the call's end) stay on the device in front of the next call's.  The host reads back a small summary per call (where the
 * records end, record and text totals), so a call returns once its work is queued behind the previous call's per-read kernels.
 * Bad magic, a header larger than max_chunk_bytes / 2, a record that fails the record check or is larger than 1 MiB, a record
 * with more than 1022 bases and a file that ends inside its header or a record are reported by vgb_sync as VGB_E_FORMAT.  CRC32
 * of the members is not verified. */
int  vgb_submit_bam(vgb_ctx *ctx, const void *comp, uint64_t comp_bytes, const vgb_bgzf_member *members, uint32_t n_members, int first, int last);
int  vgb_sync(vgb_ctx *ctx);
int  vgb_reset_counts(vgb_ctx *ctx);              /* zero the pileup counters, statistics and the trace; an unfinished gzip or BAM input goes on */
/* End the current sample: waits for all work of the context, does what vgb_reset_counts does, and drops an unfinished gzip stream
 * (bit cursor, unconsumed bytes, decode window, the text carried for records that span streams, its error) and an unfinished BAM
 * file (carried bytes, header, its error) without running or reporting them.  The index, the pinned buffers and the device
 * allocations stay.  The next submit starts a new input: a vgb_submit_gzip or vgb_submit_bam call without `first` is then
 * VGB_E_ARG.  For a cohort, one index upload serves every sample: submit, vgb_sync, vgb_call, vgb_reset_sample. */
int  vgb_reset_sample(vgb_ctx *ctx);
int  vgb_fetch_read_results(vgb_ctx *ctx, vgb_read_result *out, uint64_t cap, uint64_t *n);   /* needs VGB_CFG_TRACE */

/* ---- output VCF: replaces the rewrite of src/qv.cc:1628-1747 (the host's calls_to_map + rewrite_vcf, which stay as the
 *      reference of `vargeno-b200 vcf-rewrite`) ----
 * Output arrives in rounds through a callback: fn(user, bytes, n) gets pinned memory that is valid during the call only; it
 * returns 0 to go on (anything else ends the call with VGB_E_ARG).  Round k is handed over while the device makes round k + 1. */
typedef int (*vgb_write_fn)(void *user, const void *bytes, uint64_t n);
/* The input SNP VCF, parsed once (one scan of the bytes; records whose CHROM + POS matches no site of the uploaded index are left
 * out) and uploaded beside the index: its bytes plus about 16 B per record.  Contigs as the index's .chrlens lists them.  Needs the
 * index.  A line longer than 64 MiB is VGB_E_FORMAT.  The caller's bytes may be released when the call returns. */
int  vgb_vcf_template(vgb_ctx *ctx, const char *vcf, uint64_t nbytes, const char *const *contig_names, const uint64_t *contig_lens, uint32_t n_contigs);
/* the template of src (another context, same index) copied to dst device to device, without parsing again */
int  vgb_vcf_template_copy(vgb_ctx *dst, vgb_ctx *src);
/* One sample's VCF from its calls: gtype per site as vgb_call gives it (0 none 1 ref 2 alt 3 het) and gq per site, the
 * (int)(-1 * 10 * log(confidence)) the host computes (src/qv.cc:1681; the device never evaluates log).  The bytes are those
 * rewrite_vcf writes; with bgzf != 0 they come compressed as BGZF members (SAM specification 4.1, at most 65280 bytes of text
 * each) and the 28-byte end-of-file member.  A VCF error that depends on the sample's calls (the first failing called record,
 * as rewrite_vcf meets it) is VGB_E_FORMAT with rewrite_vcf's message, before any byte is handed over.  text_bytes (may be NULL):
 * size of the uncompressed VCF. */
int  vgb_vcf_write(vgb_ctx *ctx, const uint8_t *gtype, const int32_t *gq, uint64_t n_sites, int bgzf, vgb_write_fn fn, void *user, uint64_t *text_bytes);
/* BGZF members of any text (host memory, or device memory with text_on_device), 65280 bytes per member, then the end-of-file
 * member if eof, through fn in rounds as above */
int  vgb_deflate_bgzf(vgb_ctx *ctx, const void *text, uint64_t nbytes, int text_on_device, int eof, vgb_write_fn fn, void *user);

/* ---- probes: query_ref_dict / query_snp_dict / check_block_size / BloomFilter::check_value for a batch of
 *      packed k-mers (src/qv.cc:206-264,385-411; src/generate_bf.h:112-121) ---- */
int  vgb_lookup_kmers(vgb_ctx *ctx, const uint64_t *kmers, uint64_t n, vgb_hit *out);

/* ---- pileup + caller: replaces src/qv.cc:1573-1626 and choose_best_genotype src/qv.cc:1789-1848 ---- */
int  vgb_allreduce_pileup(vgb_ctx *ctx);          /* sum of per-GPU counters over NCCL; no-op when world_size == 1 */
int  vgb_fetch_pileup(vgb_ctx *ctx, uint32_t *ref_cnt, uint32_t *alt_cnt, uint64_t n_sites);   /* saturated at 63 (MAX_COV) */
int  vgb_call(vgb_ctx *ctx, uint8_t *gtype, double *confidence, uint64_t n_sites);             /* GTYPE_*: 0 none 1 ref 2 alt 3 het */
int  vgb_counter_device_ptr(vgb_ctx *ctx, void **ptr, uint64_t *n_u32);  /* raw device counters (2 x n_sites u32) for an external all-reduce */

int  vgb_get_stats(vgb_ctx *ctx, vgb_stats *out);

/* ---- measurement helpers (bench.py; not part of the drop-in surface) ---- */
/* n random / dictionary-sampled 32-mers generated on the device and probed against both dictionaries;
 * mode 0: uniform random (misses), 1: sampled ref-dictionary entries (hits), 2: half and half */
int  vgb_probe_bench(vgb_ctx *ctx, uint64_t n, int mode, uint64_t seed, int repeats, double *ms_per_launch, uint64_t *found);
/* uniform random 32-byte sector loads over a buffer of `bytes`: the HBM random-access roofline denominator */
int  vgb_random_sector_bench(vgb_ctx *ctx, uint64_t bytes, uint64_t n_loads, int repeats, double *gbytes_per_s);
/* synthetic FASTQ of fixed-length reads straight into device memory (twin of tools/synth.simulate_reads) */
int  vgb_synth_reads_device(vgb_ctx *ctx, const uint8_t *hap0, const uint8_t *hap1, uint64_t genome_len,
                            const uint64_t *contig_starts, const uint64_t *contig_lens, uint32_t n_contigs,
                            uint64_t n_reads, uint32_t read_len, uint64_t seed, uint64_t first_id, uint32_t id_width,
                            double sub_rate, double lowq_prob, uint32_t lowq_chars, char *device_out, uint64_t out_cap);
/* ---- index tooling on the device (SURVEY.md 8(f)-1/2, "next" rows; not part of the drop-in surface) ----
 * vgb_build_index_device: the records `vargeno index` would write (src/dictgen.c:63-275, src/generate_bf.cc:107-154,
 * 238-262), built in HBM from an upper-case ACGTN genome (device pointer, contigs concatenated) and the SNP lines that
 * survive the VCF filters (host arrays, file order; positions are 0-based in the concatenation; code = ref | alt << 2).
 * `out` receives DEVICE pointers in the on-disk record layouts; pass it to vgb_index_upload_device, copy it back with
 * vgb_memcpy_d2h to write the files, release it with vgb_free_index_device. */
int  vgb_build_index_device(vgb_ctx *ctx, const uint8_t *device_genome, uint64_t genome_len,
                            const uint64_t *contig_starts, const uint64_t *contig_lens, uint32_t n_contigs,
                            const uint32_t *snp_pos0, const uint8_t *snp_code, const uint8_t *snp_ref_freq, const uint8_t *snp_alt_freq,
                            uint64_t n_snp_lines, const uint32_t *bf_pos0, uint64_t n_bf_lines, vgb_index_view *out);
void vgb_free_index_device(vgb_ctx *ctx, vgb_index_view *view);
/* SNP Bloom filter for the UCSC snp-table input (constructBfFromUcsc, src/generate_bf.cc:439-592): 33 values per accepted record
 * (positions 0-based in the concatenation, alternative allele as a 2-bit code); words in device memory, release with vgb_device_free */
int  vgb_build_snp_bf_ucsc_device(vgb_ctx *ctx, const uint8_t *device_genome, const uint32_t *pos0, const uint8_t *alt_code, uint64_t n_lines,
                                  uint64_t **device_words, uint64_t *bits, uint64_t *nwords);
/* <prefix>.ref.bf.lite.bf, the sixth file `vargeno index` writes (src/generate_bf.cc:102-105,145-163; read by nothing): LO40 of
 * every N-free 32-mer, as sdsl bit_vector words in device memory; release with vgb_device_free */
int  vgb_build_ref_lite_bf_device(vgb_ctx *ctx, const uint8_t *device_genome, const uint64_t *contig_starts, const uint64_t *contig_lens,
                                  uint32_t n_contigs, uint64_t **device_words, uint64_t *bits, uint64_t *nwords);
int  vgb_index_upload_device(vgb_ctx *ctx, const vgb_index_view *device_view);   /* vgb_index_upload for records already in HBM */
/* random upper-case ACGT contig text, twin of tools/synth.make_genome's base layer: base i of contig c =
 * "ACGT"[(rnd64(seed, 1, c, i) >> 33) & 3] */
int  vgb_synth_genome_device(vgb_ctx *ctx, uint8_t *device_out, const uint64_t *contig_starts, const uint64_t *contig_lens,
                             uint32_t n_contigs, uint64_t seed);
void *vgb_device_alloc(vgb_ctx *ctx, uint64_t bytes);
void  vgb_device_free(vgb_ctx *ctx, void *p);
int   vgb_memcpy_d2h(vgb_ctx *ctx, void *dst, const void *src_device, uint64_t bytes);
int   vgb_memcpy_h2d(vgb_ctx *ctx, void *dst_device, const void *src, uint64_t bytes);
int   vgb_memcpy_d2d(vgb_ctx *ctx, void *dst_device, const void *src_device, uint64_t bytes);
int   vgb_memset_device(vgb_ctx *ctx, void *dst_device, int value, uint64_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* VGB200_H */
