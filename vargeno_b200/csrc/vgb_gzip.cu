// vgb_gzip.cu -- single-stream gzip FASTQ (vgb_submit_gzip) inflated on the device.
//
// The caller feeds a stream's compressed bytes in pieces of any size.  They are appended on the device behind what earlier calls
// left unconsumed, and decoded in ROUNDS: a round splits the bytes behind the exact bit cursor into sub-streams GZ_SPACING apart
// and runs the steps of vgb_gzip.cuh, one kernel each -- block finder (one thread per candidate bit), speculative decode (one warp
// per sub-stream), chain check and repair (one warp, sequential), window chain (one CTA, sequential over the sub-streams) and the
// parallel marker resolution, which writes the round's text behind the last 32 KiB of text into a chunk's text buffer.  That
// buffer then goes through the same framing and per-read kernels as a BGZF chunk, with the 32 KiB as its overlap.
//
// A round uses the sub-streams whose chain is consistent, up to the first one that ends the member, runs out of input or of
// output room; it ends at that sub-stream's last block boundary.  The host reads back a 48-byte summary per round (how much text
// there is sizes the framing launches) and a 16-byte result per member header, so a call returns once its rounds are queued
// behind the previous round's per-read kernels; per-read kernels of the last round still run when it returns.
#include <algorithm>

#include "vgb_gzip.cuh"
#include "vgb_internal.h"

namespace vgb {

#ifndef VGB_GZ_SPACING
#define VGB_GZ_SPACING 32768
#endif
constexpr uint64_t GZ_SPACING = VGB_GZ_SPACING;            // compressed bytes between the nominal starts of two sub-streams
constexpr uint32_t GZ_SLICE = 16 * VGB_GZ_SPACING;         // output symbols one sub-stream may produce (a round retries with one)
constexpr int GZ_WARPS = 4;                                // sub-streams per CTA of the decode kernel
enum { GZ_S_HEADER = 0, GZ_S_BODY = 1, GZ_S_TRAILER = 2, GZ_S_DONE = 3 };
enum { GZ_M_OK = 0, GZ_M_MORE = 1, GZ_M_NONE = 2, GZ_M_BAD = 3, GZ_M_ISIZE = 4, GZ_M_CRC = 5 };

__global__ void k_gz_init(GzSub *sub, uint32_t ns, uint64_t base)
{
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k < ns) { sub[k].start = k == 0 ? base : GZ_NONE; sub[k].status = GZ_NOSTART; sub[k].len = 0; }
}

// one thread per candidate bit of sub-streams 1 .. ns-1; the smallest bit that passes wins
__global__ void __launch_bounds__(256) k_gz_find(const uint8_t *comp, uint64_t avail, uint64_t base, uint64_t spacing_bits, uint64_t n_cand, GzSub *sub)
{
	const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n_cand) return;
	const uint64_t k = 1 + t / spacing_bits;
	const uint64_t bit = base + spacing_bits * k + t % spacing_bits;
	if (bit >= 8 * avail) return;
	if (gz_block_start(comp, avail, bit)) atomicMin(reinterpret_cast<unsigned long long *>(&sub[k].start), (unsigned long long)bit);
}

__global__ void __launch_bounds__(GZ_WARPS * 32) k_gz_decode(const uint8_t *comp, uint64_t avail, GzSub *sub, uint32_t ns, uint64_t base,
                                                             uint64_t spacing_bits, uint16_t *sym, uint32_t cap)
{
	extern __shared__ __align__(16) unsigned char gz_smem[];
	InflateWarp16 &ws = reinterpret_cast<InflateWarp16 *>(gz_smem)[threadIdx.x >> 5];
	const uint32_t k = blockIdx.x * GZ_WARPS + (threadIdx.x >> 5);
	if (k >= ns) return;
	GzSub s = sub[k];
	s.stop = gz_stop(sub, ns, k, base, spacing_bits);
	gz_decode_sub(comp, avail, s, sym + (size_t)k * cap, cap, ws);
	__syncwarp();
	if ((threadIdx.x & 31) == 0) sub[k] = s;
}

// chain check and repair: one warp walks the sub-streams in order and decodes again every one whose start the chain contradicts
__global__ void __launch_bounds__(32) k_gz_chain(const uint8_t *comp, uint64_t avail, GzSub *sub, uint32_t ns, uint16_t *sym, uint32_t cap, GzRound *round)
{
	extern __shared__ __align__(16) unsigned char gz_smem[];
	InflateWarp16 &ws = *reinterpret_cast<InflateWarp16 *>(gz_smem);
	GzRound r{};
	gz_chain(sub, ns, r, [&](uint32_t k) {
		GzSub s = sub[k];
		gz_decode_sub(comp, avail, s, sym + (size_t)k * cap, cap, ws);
		__syncwarp();
		if (threadIdx.x == 0) sub[k] = s;
		__syncwarp();
	});
	if (threadIdx.x == 0) *round = r;
}

// Window chain: the window of sub-stream k + 1 is the last 32 KiB of (window of k, text of k), in order.  One CTA; also places the
// text of every sub-stream (exclusive scan of the lengths) and leaves the last 32 KiB of the round's text in `tail`.
__global__ void __launch_bounds__(1024) k_gz_window(const uint16_t *sym, uint32_t cap, GzSub *sub, GzRound *round, uint8_t *win, uint8_t *tail,
                                                    uint32_t dec_avail, uint64_t *off)
{
	const uint32_t n = round->n_use;
	for (uint32_t i = threadIdx.x; i < INF_HIST; i += blockDim.x) win[i] = tail[i];
	__syncthreads();
	uint32_t bad = 0, av = dec_avail;
	uint64_t at = 0;
	for (uint32_t k = 0; k < n; k++) {
		const uint32_t L = sub[k].len;
		if (threadIdx.x == 0) { sub[k].win_avail = av; off[k] = at; }
		bad |= gz_window_step(sym + (size_t)k * cap, L, win + (size_t)k * INF_HIST, av, win + (size_t)(k + 1) * INF_HIST, threadIdx.x, blockDim.x);
		av = (uint32_t)min((uint64_t)INF_HIST, (uint64_t)av + L);
		at += L;
		__syncthreads();
	}
	for (uint32_t i = threadIdx.x; i < INF_HIST; i += blockDim.x) tail[i] = win[(size_t)n * INF_HIST + i];
	bad = __syncthreads_or(bad);
	if (threadIdx.x == 0) { round->text = at; round->bad_marker = bad; }
}

// every symbol of every sub-stream -> text bytes
__global__ void __launch_bounds__(256) k_gz_resolve(const uint16_t *sym, uint32_t cap, const GzSub *sub, GzRound *round, const uint8_t *win,
                                                    const uint64_t *off, uint8_t *text)
{
	const uint32_t k = blockIdx.y;
	if (k >= round->n_use) return;
	const uint32_t L = sub[k].len, av = sub[k].win_avail;
	const uint16_t *o = sym + (size_t)k * cap;
	const uint8_t *W = win + (size_t)k * INF_HIST;
	uint8_t *t = text + off[k];
	uint32_t bad = 0;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < L; i += gridDim.x * blockDim.x) t[i] = gz_resolve(o[i], W, av, bad);
	if (bad) atomicOr(&round->bad_marker, 1u);
}

// CRC-32 of each GZ_CRC_PIECE-byte piece of a round's text (one thread per piece); the host combines them in order
__global__ void __launch_bounds__(256) k_gz_crc(const uint8_t *text, uint64_t n, uint32_t *crc)
{
	__shared__ uint32_t table[256];
	table[threadIdx.x] = gz_crc_table_entry(threadIdx.x);
	__syncthreads();
	const uint64_t a = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * GZ_CRC_PIECE;
	if (a < n) crc[a / GZ_CRC_PIECE] = gz_crc_bytes(table, text + a, min((uint64_t)GZ_CRC_PIECE, n - a));
}

// the trailer of the member that just ended (ISIZE and CRC32 against its text), then the next member's header
__global__ void k_gz_member(const uint8_t *comp, uint64_t avail, uint64_t pos, int trailer, uint64_t member_text, uint32_t member_crc, uint64_t *res)
{
	uint64_t code = GZ_M_OK;
	if (trailer) {
		const int t = gz_trailer(comp + pos, avail - pos, member_text, member_crc);
		if (t) { res[0] = t == 1 ? GZ_M_MORE : t == 2 ? GZ_M_ISIZE : GZ_M_CRC; res[1] = pos; res[2] = 0; return; }
		pos += 8;
	}
	uint64_t len = 0;
	const int h = gz_member_header(comp + pos, avail - pos, &len);
	code = h == GZ_HDR_OK ? GZ_M_OK : h == GZ_HDR_MORE ? GZ_M_MORE : h == GZ_HDR_NONE ? GZ_M_NONE : GZ_M_BAD;
	res[0] = code; res[1] = pos; res[2] = len;
}

static int gz_fail(vgb_ctx *c, const char *what)
{
	GzStream &z = c->gz;
	if (!z.failed) z.err = what;
	z.failed = true;
	c->sticky_format |= 16;                                   // reported by vgb_sync as VGB_E_FORMAT
	return VGB_OK;
}

static int gz_alloc(vgb_ctx *c)
{
	GzStream &z = c->gz;
	if (z.d_comp) return VGB_OK;
	const uint64_t budget = c->max_chunk_bytes - INF_HIST - 64;
	z.max_sub = (uint32_t)std::max<uint64_t>(1, budget / GZ_SLICE);
	z.comp_cap = 2 * c->max_chunk_bytes;
	VGB_CUDA(c, cudaMalloc((void **)&z.d_comp, z.comp_cap + 64));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_sym, std::max<uint64_t>(2 * budget, c->max_chunk_bytes) + 64));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_win, (size_t)(z.max_sub + 1) * INF_HIST));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_tail, INF_HIST));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_sub, (size_t)z.max_sub * sizeof(GzSub)));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_off, (size_t)z.max_sub * sizeof(uint64_t)));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_round, sizeof(GzRound)));
	VGB_CUDA(c, cudaMalloc((void **)&z.d_member, 4 * sizeof(uint64_t)));
	const uint64_t n_piece = c->max_chunk_bytes / GZ_CRC_PIECE + 2;
	VGB_CUDA(c, cudaMalloc((void **)&z.d_crc, n_piece * sizeof(uint32_t)));
	VGB_CUDA(c, cudaMallocHost((void **)&z.h_crc, n_piece * sizeof(uint32_t)));
	VGB_CUDA(c, cudaMallocHost((void **)&z.h_round, sizeof(GzRound)));
	VGB_CUDA(c, cudaMallocHost((void **)&z.h_member, 4 * sizeof(uint64_t)));
	VGB_CUDA(c, vgb::memset_sync(c, z.d_tail, 0, INF_HIST));
	VGB_CUDA(c, cudaEventCreateWithFlags(&z.copied, cudaEventDisableTiming));
	VGB_CUDA(c, cudaEventCreateWithFlags(&z.moved, cudaEventDisableTiming));
	VGB_CUDA(c, cudaFuncSetAttribute(k_gz_decode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(GZ_WARPS * sizeof(InflateWarp16))));
	VGB_CUDA(c, cudaFuncSetAttribute(k_gz_chain, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(InflateWarp16)));
	return VGB_OK;
}

void gzip_free(vgb_ctx *c)
{
	GzStream &z = c->gz;
	cudaFree(z.d_comp); cudaFree(z.d_sym); cudaFree(z.d_win); cudaFree(z.d_tail); cudaFree(z.d_sub); cudaFree(z.d_off);
	cudaFree(z.d_round); cudaFree(z.d_member); cudaFree(z.d_crc);
	if (z.h_crc) cudaFreeHost(z.h_crc);
	if (z.h_round) cudaFreeHost(z.h_round);
	if (z.h_member) cudaFreeHost(z.h_member);
	if (z.copied) cudaEventDestroy(z.copied);
	if (z.moved) cudaEventDestroy(z.moved);
	z = GzStream();
}

void gzip_reset(vgb_ctx *c)
{
	GzStream &z = c->gz;
	z.active = false; z.failed = false; z.err.clear();
	z.state = GZ_S_HEADER; z.avail = 0; z.cur = 0; z.members = 0; z.member_text = 0; z.member_crc = 0; z.dec_avail = 0; z.tail_len = 0;
}

// One round at the cursor: ns sub-streams with `cap` output symbols each; the text goes to the next chunk slot.  *progress: the
// cursor moved.
static int gz_round(vgb_ctx *c, uint32_t ns, uint32_t cap, bool *progress)
{
	GzStream &z = c->gz;
	cudaStream_t st = c->stream;
	const uint64_t SB = 8 * GZ_SPACING;
	const int slot = c->next_slot;
	Chunk &k = c->chunk[slot];
	collect_times(c, slot);                                    // the slot's text buffer is free again
	VGB_CUDA(c, cudaEventRecord(k.t0, st));
	k_gz_init<<<(ns + 255) / 256, 256, 0, st>>>(z.d_sub, ns, z.cur);
	if (ns > 1) {
		const uint64_t n_cand = (uint64_t)(ns - 1) * SB;
		k_gz_find<<<(unsigned)((n_cand + 255) / 256), 256, 0, st>>>(z.d_comp, z.avail, z.cur, SB, n_cand, z.d_sub);
	}
	k_gz_decode<<<(ns + GZ_WARPS - 1) / GZ_WARPS, GZ_WARPS * 32, GZ_WARPS * sizeof(InflateWarp16), st>>>(z.d_comp, z.avail, z.d_sub, ns, z.cur, SB, z.d_sym, cap);
	k_gz_chain<<<1, 32, sizeof(InflateWarp16), st>>>(z.d_comp, z.avail, z.d_sub, ns, z.d_sym, cap, z.d_round);
	const uint32_t ov = z.tail_len;
	if (ov) VGB_CUDA(c, cudaMemcpyAsync(k.d_text, z.d_tail + INF_HIST - ov, ov, cudaMemcpyDeviceToDevice, st));
	k_gz_window<<<1, 1024, 0, st>>>(z.d_sym, cap, z.d_sub, z.d_round, z.d_win, z.d_tail, z.dec_avail, z.d_off);
	k_gz_resolve<<<dim3((cap + 4095) / 4096, ns), 256, 0, st>>>(z.d_sym, cap, z.d_sub, z.d_round, z.d_win, z.d_off,
	                                                            reinterpret_cast<uint8_t *>(k.d_text) + ov);
	c->launches += 5 + (ns > 1);
	VGB_CUDA(c, cudaGetLastError());
	VGB_CUDA(c, cudaMemcpyAsync(z.h_round, z.d_round, sizeof(GzRound), cudaMemcpyDeviceToHost, st));
	VGB_CUDA(c, cudaStreamSynchronize(st));
	const GzRound r = *z.h_round;
	z.subs += ns;
	z.repairs += r.repairs;
	*progress = false;
	if (r.err || r.bad_marker) return gz_fail(c, "corrupt DEFLATE data");
	if (r.text == 0 && r.end == z.cur && !r.final_block) {
		if (r.first_status == INF_E_OUTPUT && cap >= c->max_chunk_bytes - INF_HIST - 64)
			return gz_fail(c, "a DEFLATE block inflates to more than max_chunk_bytes");
		return VGB_OK;
	}
	*progress = true;
	if (r.text) {
		// CRC-32 of the round's text, in pieces, folded into the member's
		const uint64_t n_piece = (r.text + GZ_CRC_PIECE - 1) / GZ_CRC_PIECE;
		k_gz_crc<<<(unsigned)((n_piece + 255) / 256), 256, 0, st>>>(reinterpret_cast<const uint8_t *>(k.d_text) + ov, r.text, z.d_crc);
		c->launches++;
		VGB_CUDA(c, cudaGetLastError());
		VGB_CUDA(c, cudaMemcpyAsync(z.h_crc, z.d_crc, n_piece * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
		VGB_CUDA(c, cudaStreamSynchronize(st));
		const uint32_t x_piece = gz_crc_x8n(GZ_CRC_PIECE);
		for (uint64_t i = 0; i < n_piece; i++) {
			const uint64_t len = std::min<uint64_t>(GZ_CRC_PIECE, r.text - i * GZ_CRC_PIECE);
			z.member_crc = (len == GZ_CRC_PIECE ? gz_crc_mul(x_piece, z.member_crc) ^ z.h_crc[i] : gz_crc_combine(z.member_crc, z.h_crc[i], len));
		}
	}
	z.cur = r.end;
	z.member_text += r.text;
	z.dec_avail = (uint32_t)std::min<uint64_t>(INF_HIST, z.dec_avail + r.text);
	z.tail_len = (uint32_t)std::min<uint64_t>(INF_HIST, z.tail_len + r.text);
	if (r.final_block) { z.state = GZ_S_TRAILER; z.cur = (z.cur + 7) & ~7ull; }
	if (r.text == 0) return VGB_OK;
	c->next_slot ^= 1;
	return process_text(c, k, ov + r.text, 0, 1, ov, 0);
}

// Decode what the bytes at hand allow.  Without `drain` a round runs only with a full round's worth of compressed bytes (the
// rest waits for the next call); with it, everything is decoded and a stream that does not end at a member boundary is truncated.
static int gz_run(vgb_ctx *c, bool drain)
{
	GzStream &z = c->gz;
	cudaStream_t st = c->stream;
	const uint64_t budget = c->max_chunk_bytes - INF_HIST - 64;
	while (!z.failed) {
		const uint64_t at = z.cur >> 3, left = z.avail > at ? z.avail - at : 0;
		if (z.state == GZ_S_DONE) return VGB_OK;
		if (z.state != GZ_S_BODY) {
			if (left == 0) return drain && z.state == GZ_S_TRAILER ? gz_fail(c, "truncated stream (member trailer missing)") : VGB_OK;
			k_gz_member<<<1, 1, 0, st>>>(z.d_comp, z.avail, at, z.state == GZ_S_TRAILER, z.member_text, z.member_crc, z.d_member);
			c->launches++;
			VGB_CUDA(c, cudaGetLastError());
			VGB_CUDA(c, cudaMemcpyAsync(z.h_member, z.d_member, 3 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
			VGB_CUDA(c, cudaStreamSynchronize(st));
			const uint64_t code = z.h_member[0], pos = z.h_member[1];
			if (code == GZ_M_ISIZE) return gz_fail(c, "a member does not inflate to the size its trailer states");
			if (code == GZ_M_CRC) return gz_fail(c, "a member's text does not match the CRC32 of its trailer");
			if (code == GZ_M_BAD) return gz_fail(c, "bad gzip member header");
			if (pos != at) z.state = GZ_S_HEADER;              // the trailer is checked
			z.cur = 8 * pos;
			if (code == GZ_M_MORE) {
				if (z.state == GZ_S_HEADER && pos == z.avail) return VGB_OK;   // at a member boundary with no byte behind it
				return drain ? gz_fail(c, "truncated stream") : VGB_OK;
			}
			if (code == GZ_M_NONE) {
				if (!z.members) return gz_fail(c, "not a gzip stream");
				z.state = GZ_S_DONE;                           // bytes behind the last member that do not start one end the input
				continue;
			}
			z.cur = 8 * (pos + z.h_member[2]);
			z.state = GZ_S_BODY;
			z.members++;
			z.member_text = 0;
			z.member_crc = 0;
			z.dec_avail = 0;
			continue;
		}
		const uint64_t full = (uint64_t)z.max_sub * GZ_SPACING;
		if (!drain && left < full + GZ_SPACING) return VGB_OK;
		if (left == 0) return gz_fail(c, "truncated stream");
		const uint32_t ns = (uint32_t)std::min<uint64_t>(z.max_sub, (left + GZ_SPACING - 1) / GZ_SPACING);
		bool progress = false;
		int rc = gz_round(c, ns, (uint32_t)std::min<uint64_t>(GZ_SLICE, budget), &progress);
		if (rc != VGB_OK || z.failed) return rc;
		if (!progress && z.h_round->first_status == INF_E_OUTPUT) {
			rc = gz_round(c, 1, (uint32_t)budget, &progress);       // the first block needs more room than a slice
			if (rc != VGB_OK || z.failed) return rc;
		}
		if (!progress) return drain ? gz_fail(c, "truncated stream") : VGB_OK;
	}
	return VGB_OK;
}

int submit_gzip(vgb_ctx *c, const uint8_t *comp, uint64_t comp_bytes, int first, int last)
{
	if (!c->have_index) return set_err(c, VGB_E_ARG, "vgb_index_upload has not been called");
	if (comp_bytes > c->max_chunk_bytes) return set_err(c, VGB_E_ARG, "gzip piece of %llu bytes exceeds max_chunk_bytes", (unsigned long long)comp_bytes);
	cudaSetDevice(c->device);
	int rc = gz_alloc(c);
	if (rc != VGB_OK) return rc;
	GzStream &z = c->gz;
	cudaStream_t st = c->stream;
	if (first) {
		if (z.active && (rc = gz_run(c, true)) != VGB_OK) return rc;
		if (z.active && !z.failed && z.state != GZ_S_HEADER && z.state != GZ_S_DONE) gz_fail(c, "truncated stream");
		z.active = true; z.failed = false;
		z.state = GZ_S_HEADER; z.avail = 0; z.cur = 0; z.members = 0; z.member_text = 0; z.member_crc = 0; z.dec_avail = 0;   // tail_len stays: records may span streams
	}
	if (!z.active) return set_err(c, VGB_E_ARG, "vgb_submit_gzip: a stream starts with first = 1");
	if (!z.failed && z.state != GZ_S_DONE && comp_bytes) {
		if (z.avail + comp_bytes > z.comp_cap) {
			// move the bytes not consumed yet to the front (through the symbol buffer: the two ranges may overlap)
			const uint64_t at = std::min(z.cur >> 3, z.avail), keep = z.avail - at;
			if (keep) {
				VGB_CUDA(c, cudaMemcpyAsync(z.d_sym, z.d_comp + at, keep, cudaMemcpyDeviceToDevice, st));
				VGB_CUDA(c, cudaMemcpyAsync(z.d_comp, z.d_sym, keep, cudaMemcpyDeviceToDevice, st));
				VGB_CUDA(c, cudaEventRecord(z.moved, st));
				VGB_CUDA(c, cudaStreamWaitEvent(c->copy_stream, z.moved, 0));
			}
			z.cur -= 8 * at;
			z.avail = keep;
		}
		if (z.avail + comp_bytes > z.comp_cap) gz_fail(c, "a DEFLATE block needs more than max_chunk_bytes of input");
		else {
			// behind everything queued kernels read: the copy runs under them, on the copy stream
			VGB_CUDA(c, cudaMemcpyAsync(z.d_comp + z.avail, comp, comp_bytes, cudaMemcpyHostToDevice, c->copy_stream));
			VGB_CUDA(c, cudaEventRecord(z.copied, c->copy_stream));
			VGB_CUDA(c, cudaStreamWaitEvent(st, z.copied, 0));
			z.avail += comp_bytes;
		}
	}
	if ((rc = gz_run(c, last != 0)) != VGB_OK) return rc;
	if (last) {
		if (!z.failed && z.state != GZ_S_HEADER && z.state != GZ_S_DONE) gz_fail(c, "truncated stream");
		z.active = false;
		if (!z.failed && z.tail_len) {
			// the end of the input: the record that ends behind the last newline (or a truncated one) is processed here
			const int slot = c->next_slot;
			c->next_slot ^= 1;
			Chunk &k = c->chunk[slot];
			collect_times(c, slot);
			VGB_CUDA(c, cudaEventRecord(k.t0, st));
			VGB_CUDA(c, cudaMemcpyAsync(k.d_text, z.d_tail + INF_HIST - z.tail_len, z.tail_len, cudaMemcpyDeviceToDevice, st));
			if ((rc = process_text(c, k, z.tail_len, 0, 1, z.tail_len, 1)) != VGB_OK) return rc;
		}
		z.tail_len = 0;
	}
	if (comp_bytes) VGB_CUDA(c, cudaEventSynchronize(z.copied));   // the caller may reuse its buffer
	return VGB_OK;
}

}  // namespace vgb
