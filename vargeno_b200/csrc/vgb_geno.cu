// vgb_geno.cu -- the fused per-read kernel (K2 + K3 + K4): from the framed FASTQ record to the pileup, one read at a time.
//
// Replaces the body of the reference's FASTQ loop, src/qv.cc:778-1510 (SURVEY.md 3.3 is the normative
// restatement this follows):
//   encode      src/util.c:89-111 encode_kmer, reverse complement src/qv.cc:787-806
//   exact       query_ref_dict / query_snp_dict src/qv.cc:206-240,385-411; event emission :850-937
//   neighbours  Bloom gates :946-956, big-block queries :962-1109, strided small-block scan :316-376,413-464,
//               :1110-1209 (F13 kept: entry lo+S*t is examined, entry lo+t is reported), upper half :1213-1365
//   vote        improved_index_table_add :132-178 in its order-independent form (DESIGN.md section 5)
//   pileup      :1382-1502 as integer atomics on compact per-site counters (saturation deferred, SURVEY F10)
//
// The kernel is k_geno8 (vgb_geno8.inl): G lanes per read, persistent grid, 8 warps per CTA, reads claimed dynamically.  It runs
// as a chain of four stages per chunk, each over the reads the one in front handed over; this file holds the host side.
#include <cstdlib>

#include "vgb_internal.h"

namespace vgb {

constexpr int GW = 8;                 // warps per CTA

struct GEvent;                        // hit context (vgb_geno8.inl)

struct GenoArgs {
	DevIndex ix;
	const char *text;
	const uint32_t *line_start;
	uint32_t *meta;               // [1] n_reads [2] work counter [3] error bits [11] first line of the chunk's own records
	DevStats *stats;
	vgb_read_result *trace;       // nullptr unless VGB_CFG_TRACE
	GEvent *spill;                // last stage: [grid warps][EV_CAP - EV_WIDE] hit contexts behind the ones in shared memory
	uint32_t *defer;              // stages with one behind them: where reads go that need the next stage (count in meta[defer_cnt]; bit 31: start at the retry pass)
	const uint32_t *klist;        // stages behind the 4-lane one: the reads they were handed (count in meta[in_cnt]); nullptr = whole chunk
	uint32_t *kdefer;             // 4-lane stage: reads with 5..8 k-mers, for the 8-lane stage (count in meta[9])
	uint32_t in_cnt, defer_cnt;   // meta slots: in_cnt = length of klist (in_cnt + 1: its work counter), defer_cnt = length of defer
};

// reverse complement of a packed 32-mer (base b at bits 2b): reverse the base order, complement = 3 - code
__device__ __forceinline__ uint64_t revcomp64(uint64_t k)
{
	uint64_t r = __brevll(k);                                               // reverses bits: base order reversed, bit pairs swapped
	r = ((r >> 1) & 0x5555555555555555ull) | ((r & 0x5555555555555555ull) << 1);
	return ~r;
}

// the t-th substitution of base slot d: the three bases other than the current one, ascending (src/qv.cc:970-973)
__device__ __forceinline__ uint64_t substitute(uint64_t kmer, uint32_t d, uint32_t which)
{
	const uint32_t sh = 2 * d;
	const uint64_t base = (kmer >> sh) & 3ull;
	const uint64_t j = which + (which >= base ? 1 : 0);
	return (kmer & ~(3ull << sh)) | (j << sh);
}

#include "vgb_geno8.inl"

typedef void (*geno_kernel_t)(const GenoArgs);
// hit contexts + one row of counters per warp + the warp's parked reads
template <int G, int EVN>
constexpr size_t stage_smem_bytes()
{
	return sizeof(OctSmem<EVN>) * GW * (32 / G) + GW * 16 * sizeof(uint32_t) + sizeof(Pend<G>) * GW * 2 * (32 / G);
}
// the stages of the chain: 4 lanes per read, 8 lanes, 8 lanes with the wide context list, one warp per read (32 lanes)
constexpr size_t STAGE_SMEM[4] = { stage_smem_bytes<4, EV_GROUP>(), stage_smem_bytes<8, EV_GROUP>(), stage_smem_bytes<8, EV_WIDE>(),
                                   stage_smem_bytes<32, EV_WIDE>() };

int geno_prepare(vgb_ctx *c)
{
	// VGB_NO_TAIL_OVERLAP: hand-over kernels stay on the kernel stream (measurement switch); per-read results (trace) imply it
	c->tail_overlap = !(c->cfg.flags & VGB_CFG_TRACE) && !getenv("VGB_NO_TAIL_OVERLAP");
	// mean HI24 block length of the SNP dictionary decides the scan instantiation (see k_geno8): below four entries a scan ends
	// inside its first load; VGB_SHORTSCAN=0/1 overrides (measurement switch)
	bool shortscan = (c->ix.n_snp >> 24) < 4;
	if (const char *e = getenv("VGB_SHORTSCAN")) shortscan = atoi(e) != 0;
	// [stage][trace]: per-read results (VGB_CFG_TRACE: tests) are a separate instantiation, so the production kernels carry none of it
	const geno_kernel_t k[4][2] = {
		{ shortscan ? k_geno8<false, 4, EV_GROUP, true> : k_geno8<false, 4, EV_GROUP>, shortscan ? k_geno8<true, 4, EV_GROUP, true> : k_geno8<true, 4, EV_GROUP> },
		{ shortscan ? k_geno8<false, 8, EV_GROUP, true> : k_geno8<false, 8, EV_GROUP>, shortscan ? k_geno8<true, 8, EV_GROUP, true> : k_geno8<true, 8, EV_GROUP> },
		{ k_geno8<false, 8, EV_WIDE>, k_geno8<true, 8, EV_WIDE> },
		{ k_geno8<false, 32, EV_WIDE>, k_geno8<true, 32, EV_WIDE> },
	};
	for (int s = 0; s < 4; s++) {
		for (int t = 0; t < 2; t++) {
			c->grp_kernel[s][t] = (void *)k[s][t];
			VGB_CUDA(c, cudaFuncSetAttribute(k[s][t], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)STAGE_SMEM[s]));
		}
		int occ = 0;
		VGB_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k[s][0], GW * 32, STAGE_SMEM[s]));
		if (occ < 1) occ = 1;
		c->grp_grid[s] = (uint32_t)(c->sm_count * occ);
	}
	// VGB_NO_WIDE: the group stages hand their overflowing reads straight to the last one (test of the chain without the wide list)
	if (getenv("VGB_NO_WIDE")) c->grp_kernel[2][0] = c->grp_kernel[2][1] = nullptr;
	if (!c->d_spill) {
		GEvent *sp = nullptr;
		int rc = dev_alloc(c, &sp, (uint64_t)c->grp_grid[3] * GW * (EV_CAP - EV_WIDE));
		if (rc) return rc;
		c->d_spill = sp;
	}
	return VGB_OK;
}

int geno_launch(vgb_ctx *c, Chunk &ck, uint64_t nbytes, uint64_t first_read_id)
{
	(void)nbytes; (void)first_read_id;
	GenoArgs a;
	a.ix = c->ix;
	a.text = ck.d_text;
	a.line_start = ck.d_line_start;
	a.meta = ck.d_meta;
	a.stats = c->d_stats;
	a.trace = c->d_trace ? c->d_trace + c->trace_n : nullptr;
	a.spill = (GEvent *)c->d_spill;
	a.defer = ck.d_defer; a.defer_cnt = 6;
	a.klist = nullptr; a.in_cnt = 0;
	a.kdefer = ck.d_defer2;
	const int tr = a.trace ? 1 : 0;
	geno_kernel_t k[4];
	for (int s = 0; s < 4; s++) k[s] = (geno_kernel_t)c->grp_kernel[s][tr];
	// 4 lanes per read (up to 4 k-mers: 128..159 bases), then 8 lanes per read for what it handed over (5..8 k-mers), then 8
	// lanes per read with the wide context list for the reads of both with too many hit contexts, then one warp per read for
	// the rest (more than 8 k-mers, more contexts than the wide list holds)
	k[0]<<<c->grp_grid[0], GW * 32, STAGE_SMEM[0], c->stream>>>(a);
	c->launches++;
	a.klist = ck.d_defer2; a.in_cnt = 9;
	a.kdefer = nullptr;
	k[1]<<<c->grp_grid[1], GW * 32, STAGE_SMEM[1], c->stream>>>(a);
	c->launches++;
	// hand-over kernels: behind the main kernels of this chunk, and (tail_overlap) under the framing and main kernel of the next
	cudaStream_t ts = c->stream;
	ck.tail = false;
	if (c->tail_overlap) {
		VGB_CUDA(c, cudaEventRecord(ck.g1, c->stream));
		VGB_CUDA(c, cudaStreamWaitEvent(c->tail_stream, ck.g1, 0));
		VGB_CUDA(c, cudaEventRecord(ck.h0, c->tail_stream));
		ts = c->tail_stream;
		ck.tail = true;
	}
	a.klist = ck.d_defer; a.in_cnt = 6;
	if (k[2]) {
		a.defer = ck.d_defer3; a.defer_cnt = 13;
		k[2]<<<c->grp_grid[2], GW * 32, STAGE_SMEM[2], ts>>>(a);
		c->launches++;
		a.klist = ck.d_defer3; a.in_cnt = 13;
	}
	a.defer = nullptr;                // the last stage hands nothing on
	k[3]<<<c->grp_grid[3], GW * 32, STAGE_SMEM[3], ts>>>(a);
	c->launches++;
	VGB_CUDA(c, cudaGetLastError());
	return VGB_OK;
}

}  // namespace vgb
