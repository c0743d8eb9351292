// vgb_fastq.cu -- K1: FASTQ record framing on the device.
//
// Replaces the four fgets() per record of the reference (src/qv.cc:760-763): the raw text chunk is already in
// HBM; one single-pass kernel finds every line start (newline masks per 64 KiB tile, decoupled look-back for the
// running line number, scatter from registers), so the per-read kernel can address record r as lines 4r .. 4r+3
// without any host parsing.  Streaming, 128-bit loads, bounded by HBM bandwidth (the text is read ONCE + 4 B written per line).
#include <algorithm>
#include <cstdlib>

#include "vgb_inflate.cuh"
#include "vgb_internal.h"

namespace vgb {

// tile = FQ_T threads x FQ_PER bytes each (FQ_PER / 16 independent 128-bit loads per thread); default 256 x 256 B = 64 KiB

// 16-bit mask of '\n' positions among the 16 bytes at text[off .. off+16)
__device__ __forceinline__ uint32_t nl_mask16(const char *text, uint64_t off, uint64_t n, bool aligned)
{
	uint32_t m = 0;
	if (aligned && off + 16 <= n) {
		const uint4 v = __ldg(reinterpret_cast<const uint4 *>(text + off));
		const uint32_t w[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
		for (int k = 0; k < 4; k++) {
			// bytes equal to 0x0A -> bit 7 of the byte (exact zero-byte test on x = w ^ 0x0A0A0A0A), gathered by one multiply
			const uint32_t x = w[k] ^ 0x0A0A0A0Au;
			const uint32_t z = ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;
			m |= (((z >> 7) * 0x00204081u) >> 21 & 0xFu) << (4 * k);
		}
	} else {
		for (int k = 0; k < 16; k++)
			if (off + k < n && text[off + k] == '\n') m |= 1u << k;
	}
	return m;
}

// One pass over the text: tiles are claimed in order through a counter, each tile counts its newlines, publishes the
// count, learns how many newlines precede it by looking back over its predecessors' published values (decoupled
// look-back, 32 predecessors per step), and writes its line starts straight from the masks it still holds in registers.
// status[t] = flag << 32 | value: flag 0 = nothing yet, 1 = value is the tile's own count, 2 = value includes all before it.
template <int FQ_T, int FQ_PER>
__global__ void __launch_bounds__(FQ_T) k_fq_index(const char *text, uint64_t n, uint32_t n_tiles, unsigned long long *status,
                                                   uint32_t *tile_counter, uint32_t *total_nl, uint32_t *line_start, uint64_t line_cap)
{
	constexpr int FQ_NV = FQ_PER / 16;
	constexpr int FQ_TILE = FQ_T * FQ_PER;
	__shared__ uint32_t s_tile, s_prefix, sm[FQ_T / 32];
	if (threadIdx.x == 0) s_tile = atomicAdd(tile_counter, 1u);
	__syncthreads();
	const uint32_t tile = s_tile;
	const bool aligned = (reinterpret_cast<uintptr_t>(text) & 15) == 0;
	const uint64_t off = (uint64_t)tile * FQ_TILE + (uint64_t)threadIdx.x * FQ_PER;
	uint32_t m[FQ_NV / 2];                 // two 16-bit masks per word
	uint32_t cnt = 0;
#pragma unroll
	for (int k = 0; k < FQ_NV / 2; k++) {
		const uint32_t lo = off + 32 * k < n ? nl_mask16(text, off + 32 * k, n, aligned) : 0;
		const uint32_t hi = off + 32 * k + 16 < n ? nl_mask16(text, off + 32 * k + 16, n, aligned) : 0;
		m[k] = lo | (hi << 16);
		cnt += __popc(m[k]);
	}
	const uint32_t lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	uint32_t inc = cnt;
#pragma unroll
	for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
	if (lane == 31) sm[w] = inc;
	__syncthreads();
	if (w == 0) {
		uint32_t v = lane < FQ_T / 32 ? sm[lane] : 0, vi = v;
#pragma unroll
		for (int o = 1; o < FQ_T / 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, vi, o); if (lane >= (uint32_t)o) vi += t; }
		if (lane < FQ_T / 32) sm[lane] = vi - v;                       // exclusive prefix of the warp totals
		const uint32_t total = __shfl_sync(0xffffffffu, vi, FQ_T / 32 - 1);
		volatile unsigned long long *st = status;
		if (lane == 0) st[tile] = ((tile == 0 ? 2ull : 1ull) << 32) | total;
		uint32_t excl = 0;
		if (tile > 0) {
			int64_t base = (int64_t)tile - 1;
			for (;;) {
				const int64_t idx = base - lane;
				unsigned long long sv = idx >= 0 ? st[idx] : (2ull << 32);   // in front of tile 0: nothing, final
				while (__any_sync(0xffffffffu, (sv >> 32) == 0)) { if ((sv >> 32) == 0) sv = st[idx]; }
				const uint32_t fin = __ballot_sync(0xffffffffu, (sv >> 32) == 2);
				const uint32_t upto = fin ? (uint32_t)__ffs(fin) - 1 : 31u;   // nearest predecessor whose value is already a prefix
				excl += __reduce_add_sync(0xffffffffu, lane <= upto ? (uint32_t)sv : 0u);
				if (fin) break;
				base -= 32;
			}
			if (lane == 0) st[tile] = (2ull << 32) | (excl + total);
		}
		if (lane == 0) { s_prefix = excl; if (tile == n_tiles - 1) *total_nl = excl + total; }
	}
	__syncthreads();
	uint32_t idx = s_prefix + sm[w] + inc - cnt;               // newlines in front of this thread's bytes
#pragma unroll
	for (int k = 0; k < FQ_NV / 2; k++) {
		uint32_t mm = m[k];
		while (mm) {
			const int b = __ffs(mm) - 1;
			mm &= mm - 1;
			if (++idx < line_cap) line_start[idx] = (uint32_t)(off + 32 * k + b + 1);   // line idx starts right after newline idx-1
		}
	}
}

// meta: [0] n_lines [1] n_reads [2] work counter [3] format error bits [11] first line of the chunk's own records
// window (BGZF chunks, see bgzf_submit): the text starts with `ov` bytes that belong to the previous chunk (its last blocks,
// inflated again so that a record cut by the chunk boundary is whole here).  Lines are phased by the first '@' line whose second
// next line starts with '+'; the chunk owns the complete records that END behind byte ov; what is left behind the last complete
// record belongs to the next chunk (or is a truncated record when this is the last one).
__global__ void k_fq_finish(const char *text, uint64_t n, const uint32_t *total_nl, uint32_t *meta, uint32_t *line_start, uint64_t line_cap,
                            int window, uint64_t ov, int last)
{
	uint32_t lines = *total_nl;
	uint32_t err = 0, first = 0, reads = 0;
	const bool open_tail = n > 0 && text[n - 1] != '\n';   // last line without '\n': treated as terminated (end of the input only)
	if ((uint64_t)lines + 2 > line_cap) { err |= 4; lines = 0; }
	else {
		line_start[0] = 0;
		if (open_tail && (!window || last)) { line_start[lines + 1] = (uint32_t)(n + 1); lines += 1; }
	}
	if (!window) {
		if (lines % 4) err |= 1;                           // truncated record (the reference would reuse stale buffers)
		reads = lines / 4;
	} else if (lines >= 4 || (last && lines)) {
		uint32_t p = 0;
		bool found = ov == 0;                              // the first chunk starts at the beginning of the input
		for (; !found && p + 2 < lines && p < 16; p++)
			if (text[line_start[p]] == '@' && text[line_start[p + 2]] == '+') { found = true; break; }
		if (!found) err |= 1;
		else {
			const uint32_t n_rec = (lines - p) / 4;
			uint32_t j0 = 0;
			while (j0 < n_rec && (uint64_t)line_start[p + 4 * (j0 + 1)] <= ov) j0++;    // records that end inside the overlap: the previous chunk's
			first = p + 4 * j0;
			reads = n_rec - j0;
			if (last && (lines - p) % 4) err |= 1;
		}
	}
	meta[0] = lines; meta[1] = reads; meta[2] = 0; meta[3] = err; meta[6] = 0; meta[7] = 0; meta[9] = 0; meta[10] = 0; meta[11] = first; meta[13] = 0; meta[14] = 0;
	meta[5] |= err;                                        // sticky until vgb_reset_counts (the slot is reused by later chunks)
}

template <int T, int PER>
static cudaError_t launch_fq_index(Chunk &ck, uint64_t nbytes, uint64_t line_cap, cudaStream_t st)
{
	const uint64_t n_tiles = (nbytes + (uint64_t)T * PER - 1) / ((uint64_t)T * PER);
	unsigned long long *status = reinterpret_cast<unsigned long long *>(ck.d_blk_counts);   // >= max_chunk_bytes / 512 bytes
	cudaError_t e = cudaMemsetAsync(status, 0, n_tiles * sizeof(unsigned long long), st);
	if (e == cudaSuccess) e = cudaMemsetAsync(ck.d_meta + 8, 0, sizeof(uint32_t), st);    // tile counter
	if (e != cudaSuccess) return e;
	k_fq_index<T, PER><<<(unsigned)n_tiles, T, 0, st>>>(ck.d_text, nbytes, (uint32_t)n_tiles, status, ck.d_meta + 8, ck.d_meta + 4,
	                                                   ck.d_line_start, line_cap);
	return cudaSuccess;
}

int fastq_index_lines(vgb_ctx *c, Chunk &ck, uint64_t nbytes, cudaStream_t st, int window, uint64_t ov, int last)
{
	const uint64_t line_cap = c->max_chunk_bytes / 2 + 16;
	// measured on B200, 632 MB of FASTQ (profiles/r01_summary.md): 256 x 256 B 0.225 ms, 128 x 256 B 0.235, 512 x 128 B 0.262,
	// 256 x 128 B 0.267, 128 x 128 B 0.281, 1024 x 64 B 0.293 -- bytes in flight per thread matter more than the tile size
	VGB_CUDA(c, (launch_fq_index<256, 256>(ck, nbytes, line_cap, st)));
	k_fq_finish<<<1, 1, 0, st>>>(ck.d_text, nbytes, ck.d_meta + 4, ck.d_meta, ck.d_line_start, line_cap, window, ov, last);
	c->launches += 2;
	VGB_CUDA(c, cudaGetLastError());
	return VGB_OK;
}

// ---- BGZF: the gzip members of a chunk inflated on the device, one warp per member (vgb_inflate.cuh), into `out` (the chunk's
// text, or the BAM bytes of vgb_submit_bam); a corrupt member sets an error bit in the chunk's meta ----
// 7 warps of 10.6 KiB (ring + tables) per CTA, three CTAs per SM: 21 members in flight per SM.  Members are claimed one at a time
// through a counter: their cost varies with what they hold.
#ifndef VGB_INF_WARPS
#define VGB_INF_WARPS 7
#endif
constexpr int INF_WARPS = VGB_INF_WARPS;
__global__ void __launch_bounds__(INF_WARPS * 32) k_inflate_bgzf(const uint8_t *comp, const BgzfBlock *blk, uint32_t n_blk, uint8_t *out, uint32_t *meta,
                                                                 uint32_t *next_block)
{
	extern __shared__ __align__(16) unsigned char inf_smem[];
	InflateWarp &ws = reinterpret_cast<InflateWarp *>(inf_smem)[threadIdx.x >> 5];
	const uint32_t lane = threadIdx.x & 31;
	for (;;) {
		uint32_t b = 0;
		if (lane == 0) b = atomicAdd(next_block, 1u);
		b = __shfl_sync(0xffffffffu, b, 0);
		if (b >= n_blk) break;
		const BgzfBlock k = blk[b];
		uint32_t got = 0;
		const int rc = inflate_block(comp + k.comp_off, k.comp_len, out + k.out_off, k.out_len, ws, &got);
		if (lane == 0 && (rc != INF_OK || got != k.out_len)) atomicOr(&meta[5], 8u);   // corrupt member: sticky, reported by vgb_sync
		__syncwarp();
	}
}

int bgzf_inflate(vgb_ctx *c, Chunk &ck, const uint8_t *d_comp, const BgzfBlock *d_blk, uint32_t n_blk, cudaStream_t st, uint8_t *out)
{
	const size_t smem = sizeof(InflateWarp) * INF_WARPS;
	if (!c->inflate_ready) {
		int occ = 0;
		VGB_CUDA(c, cudaFuncSetAttribute(k_inflate_bgzf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		VGB_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_inflate_bgzf, INF_WARPS * 32, smem));
		c->inflate_grid = (uint32_t)(c->sm_count * (occ > 0 ? occ : 1));
		c->inflate_ready = true;
	}
	VGB_CUDA(c, cudaMemsetAsync(ck.d_meta + 12, 0, sizeof(uint32_t), st));                // member counter
	const unsigned grid = (unsigned)std::min<uint64_t>(c->inflate_grid, (n_blk + INF_WARPS - 1) / INF_WARPS);
	k_inflate_bgzf<<<grid ? grid : 1, INF_WARPS * 32, smem, st>>>(d_comp, d_blk, n_blk, out, ck.d_meta, ck.d_meta + 12);
	c->launches++;
	VGB_CUDA(c, cudaGetLastError());
	return VGB_OK;
}

}  // namespace vgb
