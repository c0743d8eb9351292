// vgb_internal.h -- host-side context shared by the translation units of libvgb200.so
#pragma once
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>

#include <cuda_runtime.h>

#include "../../include/vgb200.h"
#include "vgb_common.cuh"

namespace vgb {

struct DevStats {   // device-resident counters, one cache line apart from nothing important; fetched by vgb_get_stats
	unsigned long long reads, skipped_n, passes, placed, exact_lookups, nbr_query_lookups, nbr_scan_reads, bf_probes,
	    lowq_kmers, events, pileup_incr, big_kmers, bad_records, overflow_reads, freq_wrap_reads, first_error;
};

struct BgzfBlock { uint32_t comp_off, comp_len, out_off, out_len; };   // one gzip member of a chunk: DEFLATE payload in the compressed buffer -> place in the text

struct Chunk {          // one in-flight FASTQ chunk (two slots: copy of chunk i+1 overlaps the kernels of chunk i)
	char *d_text = nullptr;           // device copy of the text (owned unless external)
	char *h_pinned = nullptr;         // pinned staging buffer handed out by vgb_pinned_buffer
	uint32_t *d_line_start = nullptr; // [max_lines + 1] byte offset of each line start
	uint32_t *d_blk_counts = nullptr; // newline count per 4 KiB tile, then its exclusive scan
	uint32_t *d_defer = nullptr;      // read indices the 4- and 8-lane kernels hand to the wide-list kernel (or the last one)
	uint32_t *d_defer2 = nullptr;     // read indices the 4-lane kernel hands to the 8-lane kernel
	uint32_t *d_defer3 = nullptr;     // read indices the wide-list kernel hands to the one-warp-per-read kernel
	uint8_t *d_comp = nullptr;        // BGZF: compressed members of the chunk (allocated at the first vgb_submit_bgzf)
	BgzfBlock *d_blk = nullptr, *h_blk = nullptr;   // their table, device copy and pinned staging
	uint32_t blk_cap = 0;
	uint32_t *d_meta = nullptr;       // [0] n_lines [1] n_reads [2] work counter [3] format error [5] sticky errors [6] deferred reads [7] their work counter [8] framing tile counter [9] reads for the 8-lane kernel [10] their work counter [11] first line of the chunk's own records [12] BGZF member counter [13] reads for the one-warp-per-read kernel [14] their work counter
	cudaEvent_t copied = nullptr, done = nullptr, t0 = nullptr, t1 = nullptr, g0 = nullptr;
	cudaEvent_t g1 = nullptr, h0 = nullptr;   // end of the main kernels on the kernel stream, start of the hand-over kernels on the tail stream
	bool tail = false;                        // this chunk's hand-over kernels went to the tail stream (`done` is recorded there)
	bool busy = false;
};

}  // namespace vgb

struct vgb_ctx {
	vgb_config cfg{};
	int device = 0;
	int sm_count = 148;
	cudaStream_t stream = nullptr, copy_stream = nullptr;   // kernels | H2D copies (chunk i+1 is copied under the kernels of chunk i)
	// The hand-over kernels of a chunk (wide-list stage, one-warp-per-read stage: a few thousand reads from repeat families, a long
	// dependent chain each, the GPU mostly idle) run here, under the framing and the main kernel of the NEXT chunk.  Not in trace mode.
	cudaStream_t tail_stream = nullptr;
	bool tail_overlap = false;
	std::string err;

	// index (device)
	vgb::DevIndex ix{};
	bool have_index = false;
	uint32_t *d_site_pos = nullptr;
	uint8_t *d_site_rf = nullptr, *d_site_af = nullptr;
	double *d_tables = nullptr;      // g[64][64][3] then poisson[127]
	void *owned[64] = {};            // device allocations freed at destroy
	int n_owned = 0;

	// reads
	uint64_t max_chunk_bytes = 0;
	vgb::Chunk chunk[2];
	int next_slot = 0;
	vgb::DevStats *d_stats = nullptr;
	vgb_read_result *d_trace = nullptr;
	uint64_t trace_cap = 0, trace_n = 0;
	uint32_t sticky_format = 0;      // format error bits seen since the last reset
	bool upload_from_device = false; // vgb_index_upload_device: the index view holds device pointers
	void *d_spill = nullptr;         // per-warp overflow area for hit contexts of the last stage
	uint8_t *d_call_gt = nullptr;    // per-site output staging of vgb_call / vgb_fetch_pileup (allocated once, at first use)
	double *d_call_conf = nullptr;
	uint32_t *d_fetch_ref = nullptr, *d_fetch_alt = nullptr;
	// kernel choice of this context (geno_prepare): instantiation + persistent grid per stage; nothing process-wide
	void *grp_kernel[4][2] = {};     // [0: 4 lanes per read, 1: 8 lanes, 2: 8 lanes with the wide context list (nullptr: VGB_NO_WIDE), 3: 32 lanes][trace]
	uint32_t grp_grid[4] = {};
	bool inflate_ready = false;       // k_inflate_bgzf: shared-memory attribute set, grid sized
	uint32_t inflate_grid = 0;

	// host-side statistics
	uint64_t chunks = 0, chunk_bytes = 0, launches = 0;
	double ms_parse = 0, ms_geno = 0;
	cudaEvent_t ev[4] = {};

	// NCCL (dlopen)
	void *nccl_comm = nullptr;
	unsigned char uid[128] = {};     // copy of the unique id handed to vgb_comm_init
};

namespace vgb {

int set_err(vgb_ctx *c, int code, const char *fmt, ...);
extern thread_local std::string g_create_err;

#define VGB_CUDA(c, call)                                                                        \
	do {                                                                                         \
		cudaError_t e__ = (call);                                                                \
		if (e__ != cudaSuccess)                                                                  \
			return vgb::set_err((c), VGB_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
	} while (0)

// Host-blocking copy / fill ORDERED ON THE CONTEXT'S KERNEL STREAM.  c->stream is created cudaStreamNonBlocking, so the
// legacy-default-stream forms (cudaMemcpy / cudaMemset) are not ordered with the kernels at all: a pageable H2D copy may
// return before its last DMA lands and a device memset returns before it ran.  Everything the library copies or clears
// goes through these two.
inline cudaError_t copy_sync(vgb_ctx *c, void *dst, const void *src, size_t n, cudaMemcpyKind kind)
{
	cudaError_t e = cudaMemcpyAsync(dst, src, n, kind, c->stream);
	if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
	return e;
}
inline cudaError_t memset_sync(vgb_ctx *c, void *dst, int value, size_t n)
{
	cudaError_t e = cudaMemsetAsync(dst, value, n, c->stream);
	if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
	return e;
}

template <typename T>
int dev_alloc(vgb_ctx *c, T **p, uint64_t count, bool own = true)
{
	void *q = nullptr;
	cudaError_t e = cudaMalloc(&q, (count ? count : 1) * sizeof(T));
	if (e != cudaSuccess) return set_err(c, VGB_E_CUDA, "cudaMalloc(%llu bytes) failed: %s", (unsigned long long)(count * sizeof(T)), cudaGetErrorString(e));
	*p = (T *)q;
	if (own && c->n_owned < 64) c->owned[c->n_owned++] = q;
	return VGB_OK;
}

// vgb_index.cu
int index_upload(vgb_ctx *c, const vgb_index_view *v);
// vgb_fastq.cu
int fastq_index_lines(vgb_ctx *c, Chunk &ck, uint64_t nbytes, cudaStream_t st, int window = 0, uint64_t ov = 0, int last = 0);
int bgzf_inflate(vgb_ctx *c, Chunk &ck, const uint8_t *d_comp, const BgzfBlock *d_blk, uint32_t n_blk, cudaStream_t st);
// vgb_geno.cu
int geno_launch(vgb_ctx *c, Chunk &ck, uint64_t nbytes, uint64_t first_read_id);
int geno_prepare(vgb_ctx *c);
// vgb_call.cu
int call_sites(vgb_ctx *c, uint8_t *gtype, double *conf, uint64_t n_sites);
int fetch_pileup(vgb_ctx *c, uint32_t *ref_cnt, uint32_t *alt_cnt, uint64_t n_sites);
void build_call_tables(double *g /*64*64*3*/, double *poisson /*127*/);   // vgb_tables.cpp (plain C++, glibc libm)
// vgb_bench.cu
int lookup_kmers(vgb_ctx *c, const uint64_t *kmers, uint64_t n, vgb_hit *out);
int probe_bench(vgb_ctx *c, uint64_t n, int mode, uint64_t seed, int repeats, double *ms, uint64_t *found);
int random_sector_bench(vgb_ctx *c, uint64_t bytes, uint64_t n_loads, int repeats, double *gbs);
int synth_reads(vgb_ctx *c, const uint8_t *hap0, const uint8_t *hap1, uint64_t genome_len, const uint64_t *cstart,
                const uint64_t *clen, uint32_t n_contigs, uint64_t n_reads, uint32_t read_len, uint64_t seed, uint64_t first_id,
                uint32_t id_width, double sub_rate, double lowq_prob, uint32_t lowq_chars, char *out, uint64_t out_cap);
// vgb_build.cu
int build_index_device(vgb_ctx *c, const uint8_t *d_genome, uint64_t genome_len, const uint64_t *cstart, const uint64_t *clen, uint32_t n_contigs,
                       const uint32_t *snp_pos0, const uint8_t *snp_code, const uint8_t *snp_rf, const uint8_t *snp_af, uint64_t n_snp_lines,
                       const uint32_t *bf_pos0, uint64_t n_bf_lines, vgb_index_view *out);
void free_index_device(vgb_index_view *v);
int build_snp_bf_ucsc(vgb_ctx *c, const uint8_t *d_genome, const uint32_t *pos0, const uint8_t *alt, uint64_t n, uint64_t **d_words, uint64_t *bits, uint64_t *nwords);
int build_ref_lite_bf(vgb_ctx *c, const uint8_t *d_genome, const uint64_t *cstart, const uint64_t *clen, uint32_t n_contigs,
                      uint64_t **d_words, uint64_t *bits, uint64_t *nwords);
int synth_genome(vgb_ctx *c, uint8_t *d_out, const uint64_t *cstart, const uint64_t *clen, uint32_t n_contigs, uint64_t seed);
// vgb_nccl.cpp
int nccl_unique_id(void *out128, std::string &err);
int nccl_init(vgb_ctx *c);
int nccl_allreduce_u32(vgb_ctx *c, uint32_t *buf, uint64_t n);
void nccl_destroy(vgb_ctx *c);

// generic device exclusive scan over uint32 (vgb_scan.cuh users): out[i] = sum_{j<i} in[j]; returns total through d_total
int exclusive_scan_u32(vgb_ctx *c, const uint32_t *d_in, uint32_t *d_out, uint64_t n, uint32_t *d_tmp /* >= n/2048+2 */, uint32_t *d_total);

}  // namespace vgb
