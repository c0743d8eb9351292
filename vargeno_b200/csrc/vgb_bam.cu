// vgb_bam.cu -- BAM input (vgb_submit_bam): BGZF members inflated on the device, records framed and written out as FASTQ text
// on the device, then the same framing and per-read kernels as any FASTQ chunk.
//
// A call's members are inflated (k_inflate_bgzf) behind the bytes the previous call did not consume -- a header that is not
// complete yet or the record cut by the end of the previous call -- into one of two BAM buffers; the bytes this call leaves go to
// the front of the other one.  The header is parsed on the device at the first call of a file.  The records are then framed by
// the steps of vgb_bam.cuh, one kernel each -- speculate and walk (one warp per tile), chain check and repair (one thread), the
// scans of the tiles' record counts and text sizes, the record list (one thread per tile) and the round plan -- and the host reads
// back a small summary (BamSum: where the chain ended, record and text totals, round boundaries).  Each round writes its records
// into a chunk's text buffer (one warp per record) and hands it to process_text.  So a call returns once its rounds are queued
// behind the previous call's per-read kernels.
#include <algorithm>

#include "vgb_bam.cuh"
#include "vgb_internal.h"

namespace vgb {

constexpr int BAM_WARPS = 8;                                // tiles per CTA of the speculate kernel, records per CTA of the convert kernel

// one warp per tile: tile 0 starts at the first record; every other tile at the first offset that passes the record check (a
// warp checks 32 offsets at a time).  Then lane 0 walks the tile.
__global__ void __launch_bounds__(BAM_WARPS * 32) k_bam_spec(const uint8_t *p, uint32_t n, uint32_t first, uint32_t nt, int32_t n_ref, BamTile *tile)
{
	const uint32_t k = blockIdx.x * BAM_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
	if (k >= nt) return;
	const uint32_t a = first + k * BAM_TILE, b = (uint32_t)min((uint64_t)a + BAM_TILE, (uint64_t)n);
	uint32_t start = k == 0 ? first : BAM_NONE;
	for (uint32_t base = a; k && base < b; base += 32) {
		const uint32_t o = base + lane;
		const uint32_t hit = __ballot_sync(0xffffffffu, o < b && bam_check(p, n, o, n_ref) == BAM_REC_YES);
		if (hit) { start = base + __ffs(hit) - 1; break; }
	}
	if (lane == 0) {
		BamTile t;
		t.start = start;
		bam_walk(p, n, n_ref, a + BAM_TILE, t);
		tile[k] = t;
	}
}

// chain check and repair (thread 0, in tile order), then every thread writes the tiles' record counts and text sizes for the scans
__global__ void __launch_bounds__(256) k_bam_chain(const uint8_t *p, uint32_t n, uint32_t first, uint32_t nt, int32_t n_ref, BamTile *tile,
                                                   uint32_t *cnt, uint32_t *txt, BamSum *sum)
{
	__shared__ uint32_t s_use;
	if (threadIdx.x == 0) {
		BamSum r = *sum;
		bam_chain(tile, nt, first, r, [&](uint32_t k) { bam_walk(p, n, n_ref, first + k * BAM_TILE + BAM_TILE, tile[k]); });
		*sum = r;
		s_use = r.n_use;
	}
	__syncthreads();
	for (uint32_t k = threadIdx.x; k < nt; k += blockDim.x) {
		const bool use = k < s_use;
		cnt[k] = use ? tile[k].n_rec : 0;
		txt[k] = use ? tile[k].text : 0;
	}
}

// one thread per chained tile: the offsets of its FASTQ records and of their text (cnt, txt: exclusive scans over the tiles)
__global__ void __launch_bounds__(256) k_bam_list(const uint8_t *p, const BamTile *tile, const BamSum *sum, const uint32_t *cnt, const uint32_t *txt,
                                                  uint32_t *rec_off, uint32_t *rec_txt)
{
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k < sum->n_use) bam_list(p, tile[k], cnt[k], txt[k], rec_off, rec_txt);
}

__global__ void k_bam_plan(const uint32_t *rec_txt, BamSum *sum, uint32_t cap)
{
	bam_plan(rec_txt, *sum, cap);                          // in place: the round arrays are indexed dynamically
}

__global__ void k_bam_header(const uint8_t *p, uint32_t n, BamSum *sum)
{
	uint64_t len = 0;
	int32_t n_ref = 0;
	const int h = bam_header(p, n, &len, &n_ref);
	sum->hdr_code = (uint32_t)h;
	sum->hdr_len = (uint32_t)min(len, (uint64_t)n);
	sum->n_ref = n_ref;
}

// one warp per FASTQ record of records [r0, r1): its text at rec_txt[i] - text_base of `out`
__global__ void __launch_bounds__(BAM_WARPS * 32) k_bam_convert(const uint8_t *p, const uint32_t *rec_off, const uint32_t *rec_txt, uint32_t r0, uint32_t r1,
                                                                uint32_t text_base, char *out)
{
	const uint32_t i = r0 + blockIdx.x * BAM_WARPS + (threadIdx.x >> 5);
	if (i >= r1) return;
	bam_emit(p + rec_off[i], out + (rec_txt[i] - text_base), threadIdx.x & 31, 32);
}

static int bam_fail(vgb_ctx *c, const char *what)
{
	BamStream &z = c->bam;
	if (!z.failed) z.err = what;
	z.failed = true;
	c->sticky_format |= 32;                                   // reported by vgb_sync as VGB_E_FORMAT
	return VGB_OK;
}

static int bam_alloc(vgb_ctx *c)
{
	BamStream &z = c->bam;
	if (z.d_buf[0]) return VGB_OK;
	// unconsumed bytes: a header of at most max_chunk_bytes / 2 or one cut record
	z.cap = c->max_chunk_bytes + std::max<uint64_t>(c->max_chunk_bytes / 2, 4 + BAM_REC_MAX) + 64;
	z.max_tiles = (uint32_t)(z.cap / BAM_TILE + 2);
	const uint64_t max_rec = z.cap / 37 + 16;                 // a record takes at least 37 bytes
	for (int i = 0; i < 2; i++) VGB_CUDA(c, cudaMalloc((void **)&z.d_buf[i], z.cap));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_tile, (size_t)z.max_tiles * sizeof(BamTile)));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_cnt, (size_t)z.max_tiles * 4));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_txt, (size_t)z.max_tiles * 4));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_scan, (size_t)(z.max_tiles / 2048 + 8) * 4));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_rec_off, max_rec * 4));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_rec_txt, max_rec * 4));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_sum, sizeof(BamSum)));
	VGB_CUDA(c, cudaMallocHost((void **)&z.h_sum, sizeof(BamSum)));
	return VGB_OK;
}

void bam_free(vgb_ctx *c)
{
	BamStream &z = c->bam;
	cudaFree(z.d_buf[0]); cudaFree(z.d_buf[1]); cudaFree(z.d_tile); cudaFree(z.d_cnt); cudaFree(z.d_txt); cudaFree(z.d_scan);
	cudaFree(z.d_rec_off); cudaFree(z.d_rec_txt); cudaFree(z.d_sum);
	if (z.h_sum) cudaFreeHost(z.h_sum);
	z = BamStream();
}

void bam_reset(vgb_ctx *c)
{
	BamStream &z = c->bam;
	z.active = false; z.failed = false; z.err.clear();
	z.header_done = false; z.carry = 0; z.n_ref = 0; z.cur = 0; z.long_records = 0;
}

static int bam_readback(vgb_ctx *c)
{
	BamStream &z = c->bam;
	VGB_CUDA(c, cudaMemcpyAsync(z.h_sum, z.d_sum, sizeof(BamSum), cudaMemcpyDeviceToHost, c->stream));
	VGB_CUDA(c, cudaStreamSynchronize(c->stream));
	return VGB_OK;
}

// the n bytes at the front of the current buffer: header (first call of a file), framing, conversion rounds; the bytes behind what
// was consumed go to the front of the other buffer
static int bam_frame(vgb_ctx *c, uint32_t n)
{
	BamStream &z = c->bam;
	cudaStream_t st = c->stream;
	const uint8_t *buf = z.d_buf[z.cur];
	uint32_t first = 0, keep = n;
	int rc;
	VGB_CUDA(c, cudaMemsetAsync(z.d_sum, 0, sizeof(BamSum), st));
	if (!z.header_done && n) {
		k_bam_header<<<1, 1, 0, st>>>(buf, n, z.d_sum);
		c->launches++;
		VGB_CUDA(c, cudaGetLastError());
		if ((rc = bam_readback(c)) != VGB_OK) return rc;
		const BamSum &h = *z.h_sum;
		if (h.hdr_code == BAM_HDR_BAD) return bam_fail(c, "not a BAM file (bad magic) or a corrupt header");
		if (h.hdr_code == BAM_HDR_OK) {
			z.header_done = true;
			z.n_ref = h.n_ref;
			first = h.hdr_len;
			keep = n - first;
		}
		if ((h.hdr_code == BAM_HDR_OK ? h.hdr_len : n) > c->max_chunk_bytes / 2) return bam_fail(c, "the header is larger than max_chunk_bytes / 2");
	}
	if (z.header_done && n > first) {
		const uint32_t nt = (n - first + BAM_TILE - 1) / BAM_TILE;
		k_bam_spec<<<(nt + BAM_WARPS - 1) / BAM_WARPS, BAM_WARPS * 32, 0, st>>>(buf, n, first, nt, z.n_ref, z.d_tile);
		k_bam_chain<<<1, 256, 0, st>>>(buf, n, first, nt, z.n_ref, z.d_tile, z.d_cnt, z.d_txt, z.d_sum);
		c->launches += 2;
		VGB_CUDA(c, cudaGetLastError());
		if ((rc = exclusive_scan_u32(c, z.d_cnt, z.d_cnt, nt, z.d_scan, &z.d_sum->n_rec)) != VGB_OK) return rc;
		if ((rc = exclusive_scan_u32(c, z.d_txt, z.d_txt, nt, z.d_scan, &z.d_sum->text)) != VGB_OK) return rc;
		k_bam_list<<<(nt + 255) / 256, 256, 0, st>>>(buf, z.d_tile, z.d_sum, z.d_cnt, z.d_txt, z.d_rec_off, z.d_rec_txt);
		k_bam_plan<<<1, 1, 0, st>>>(z.d_rec_txt, z.d_sum, (uint32_t)c->max_chunk_bytes);
		c->launches += 2;
		VGB_CUDA(c, cudaGetLastError());
		if ((rc = bam_readback(c)) != VGB_OK) return rc;
		const BamSum s = *z.h_sum;
		z.tiles += nt;
		z.repairs += s.repairs;
		z.long_records += s.n_long;
		if (s.status == BAM_W_BAD) return bam_fail(c, "a record fails the record check (block_size, refID, name or field sizes)");
		if (s.status == BAM_W_BIG) return bam_fail(c, "a record is larger than 1 MiB");
		if (s.n_long) bam_fail(c, "a record has more than 1022 bases (the FASTQ line limit)");
		if (s.n_rec && !s.n_round) return bam_fail(c, "the records of one call convert to more text than the rounds hold");
		for (uint32_t r = 0; r < s.n_round; r++) {
			const uint32_t r0 = s.round[r], r1 = s.round[r + 1];
			const int slot = c->next_slot;
			c->next_slot ^= 1;
			Chunk &k = c->chunk[slot];
			collect_times(c, slot);                           // the slot's text buffer is free again
			const uint32_t base = s.round_txt[r], end = s.round_txt[r + 1];
			k_bam_convert<<<(r1 - r0 + BAM_WARPS - 1) / BAM_WARPS, BAM_WARPS * 32, 0, st>>>(buf, z.d_rec_off, z.d_rec_txt, r0, r1, base, k.d_text);
			c->launches++;
			VGB_CUDA(c, cudaGetLastError());
			if ((rc = process_text(c, k, end - base, 0, 0, 0, 0)) != VGB_OK) return rc;
		}
		keep = n - s.end;
	}
	if (keep) VGB_CUDA(c, cudaMemcpyAsync(z.d_buf[z.cur ^ 1], buf + (n - keep), keep, cudaMemcpyDeviceToDevice, st));
	z.cur ^= 1;
	z.carry = keep;
	return VGB_OK;
}

int submit_bam(vgb_ctx *c, const uint8_t *comp, uint64_t comp_bytes, const vgb_bgzf_member *mem, uint32_t n_mem, int first, int last)
{
	if (!c->have_index) return set_err(c, VGB_E_ARG, "vgb_index_upload has not been called");
	if (c->max_chunk_bytes > (1ull << 30)) return set_err(c, VGB_E_ARG, "BAM input needs max_chunk_bytes <= 1 GiB (32-bit offsets into a call's records)");
	cudaSetDevice(c->device);
	int rc = bam_alloc(c);
	if (rc != VGB_OK) return rc;
	BamStream &z = c->bam;
	if (first) {
		if (z.active && !z.failed && (z.carry || !z.header_done)) bam_fail(c, "truncated file (a header or a record is cut)");
		z.active = true; z.failed = false; z.header_done = false; z.carry = 0; z.n_ref = 0;
	}
	if (!z.active) return set_err(c, VGB_E_ARG, "vgb_submit_bam: a file starts with first = 1");
	if (!z.failed) {
		const int slot = c->next_slot;
		Chunk &k = c->chunk[slot];
		collect_times(c, slot);
		uint64_t out = 0;
		if ((rc = bgzf_stage(c, k, slot, comp, comp_bytes, mem, n_mem, &out)) != VGB_OK) return rc;
		if (out && (rc = bgzf_inflate(c, k, k.d_comp, k.d_blk, n_mem, c->stream, z.d_buf[z.cur] + z.carry)) != VGB_OK) return rc;
		if ((rc = bam_frame(c, (uint32_t)(z.carry + out))) != VGB_OK) return rc;
	}
	if (last) {
		if (!z.failed && (z.carry || !z.header_done)) bam_fail(c, "truncated file (a header or a record is cut)");
		z.active = false;
		z.carry = 0;
	}
	return VGB_OK;
}

}  // namespace vgb
