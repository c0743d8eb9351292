// vgb_vcf.cu -- the output VCF on the device (vgb_vcf_template, vgb_vcf_template_copy, vgb_vcf_write) and the BGZF writer
// (vgb_deflate_bgzf).  The splice rules are in vgb_vcf.cuh, the compressor in vgb_deflate.cuh; both also compile for the host.
//
// Per sample: the calls (one gtype byte and one GQ int32 per site) are uploaded; k_vcf_first finds the first called record that
// takes its GT index from FORMAT and k_vcf_gi reads that index; k_vcf_size computes every record's output length and the first
// failing record; the lengths are scanned into 64-bit offsets (k_scan64_*).  The output is then made in rounds of VCF_ROUND bytes: k_vcf_write (one warp per
// record, lane 0 plans, the lanes write the bytes) fills the round's text; for BGZF, k_deflate compresses it one warp per
// 65280-byte block, the member sizes are scanned and k_member_compact packs the members.  One copy back per round, into two
// pinned buffers in turn: the caller's callback gets round k while the device makes round k + 1.
#include <algorithm>
#include <vector>

#include "vgb_internal.h"
#include "vgb_deflate.cuh"
#include "vgb_vcf.cuh"

namespace vgb {

constexpr uint32_t VCF_BLOCKS = 1024;                               // BGZF blocks per round
constexpr uint64_t VCF_ROUND = (uint64_t)VCF_BLOCKS * DF_BLOCK;     // text bytes per round
constexpr uint64_t VCF_OUT_CAP = (uint64_t)VCF_BLOCKS * DF_MEMBER_MAX;
constexpr int VCF_WARPS = 8;                                        // warps per block of k_vcf_write

enum { M_ERR = 0, M_FIRST = 1, M_GI = 2, M_TOTAL = 3, M_OUT = 4 };  // d_misc words

__global__ void __launch_bounds__(256) k_vcf_first(const VcfRec *rec, uint64_t n, const uint32_t *lists, const uint8_t *gt, unsigned long long *misc)
{
	const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n) return;
	const uint32_t f = rec[r].len_flags;
	if ((f & VCF_LIT) || !(f & VCF_HAS_GT) || (f & VCF_GT0)) return;
	if (vcf_site(lists, rec[r].list, gt) >= 0) atomicMin(&misc[M_FIRST], (unsigned long long)r);
}

__global__ void k_vcf_gi(const VcfRec *rec, const uint8_t *text, unsigned long long *misc)
{
	const unsigned long long r = misc[M_FIRST];
	misc[M_GI] = (unsigned long long)(long long)(r == ~0ull ? -1 : vcf_find_gt(text + rec[r].off, rec[r].len_flags & VCF_LEN_MASK, rec[r].len_flags));
}

__global__ void __launch_bounds__(256) k_vcf_size(const VcfRec *rec, uint64_t n, const uint32_t *lists, const uint8_t *gt, const int32_t *gq,
                                                  const uint8_t *text, unsigned long long *misc, uint32_t *len)
{
	const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	uint64_t m = 0;
	if (r < n) {
		const VcfRec x = rec[r];
		const uint32_t l = x.len_flags & VCF_LEN_MASK;
		if (x.len_flags & VCF_LIT) m = l;
		else {
			const int64_t s = vcf_site(lists, x.list, gt);
			if (s >= 0) {
				const int64_t v = vcf_plan<false>(text + x.off, l, x.len_flags, gt[s], gq[s], (int32_t)(long long)misc[M_GI], nullptr);
				if (v < 0) atomicMin(&misc[M_ERR], (unsigned long long)(r << 3 | (uint64_t)-v));
				else m = (uint64_t)v;
			}
		}
		len[r] = (uint32_t)m;
	}
	for (int o = 16; o; o >>= 1) m += __shfl_xor_sync(0xffffffffu, m, o);
	if ((threadIdx.x & 31) == 0 && m) atomicAdd(&misc[M_TOTAL], (unsigned long long)m);
}

// ---- exclusive scan of the u32 record lengths into u64 offsets (an output VCF may pass 4 GiB): tile sums, one CTA over the
// tiles, then each tile again from its base ----
constexpr int S64_T = 256, S64_I = 8;
constexpr uint64_t S64_TILE = (uint64_t)S64_T * S64_I;

// exclusive scan of v over the CTA (blockDim.x = S64_T or 1024); sm: 32 words
__device__ uint64_t block_scan64(uint64_t v, uint64_t *total, uint64_t *sm)
{
	const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
	uint64_t x = v;
	for (int o = 1; o < 32; o <<= 1) { const uint64_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
	if (lane == 31) sm[wid] = x;
	__syncthreads();
	if (wid == 0) {
		uint64_t t = lane < nw ? sm[lane] : 0;
		for (int o = 1; o < 32; o <<= 1) { const uint64_t y = __shfl_up_sync(0xffffffffu, t, o); if (lane >= o) t += y; }
		sm[lane] = t;
	}
	__syncthreads();
	const uint64_t r = (wid ? sm[wid - 1] : 0) + x - v;
	if (total) *total = sm[nw - 1];
	__syncthreads();
	return r;
}

__global__ void __launch_bounds__(S64_T) k_scan64_tiles(const uint32_t *in, uint64_t n, uint64_t *tsum)
{
	__shared__ uint64_t sm[32];
	const uint64_t base = (uint64_t)blockIdx.x * S64_TILE + (uint64_t)threadIdx.x * S64_I;
	uint64_t s = 0;
	for (int i = 0; i < S64_I; i++) if (base + i < n) s += in[base + i];
	uint64_t tot;
	block_scan64(s, &tot, sm);
	if (threadIdx.x == 0) tsum[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(1024) k_scan64_top(uint64_t *tsum, uint64_t nt)
{
	__shared__ uint64_t sm[32];
	uint64_t carry = 0;
	for (uint64_t b = 0; b < nt; b += 1024) {
		const uint64_t j = b + threadIdx.x;
		const uint64_t v = j < nt ? tsum[j] : 0;
		uint64_t tot;
		const uint64_t ex = block_scan64(v, &tot, sm);
		if (j < nt) tsum[j] = carry + ex;
		carry += tot;
	}
}

__global__ void __launch_bounds__(S64_T) k_scan64_apply(const uint32_t *in, uint64_t n, const uint64_t *tsum, uint64_t *out)
{
	__shared__ uint64_t sm[32];
	const uint64_t base = (uint64_t)blockIdx.x * S64_TILE + (uint64_t)threadIdx.x * S64_I;
	uint32_t v[S64_I];
	uint64_t s = 0;
#pragma unroll
	for (int i = 0; i < S64_I; i++) { v[i] = base + i < n ? in[base + i] : 0; s += v[i]; }
	uint64_t run = block_scan64(s, nullptr, sm) + tsum[blockIdx.x];
#pragma unroll
	for (int i = 0; i < S64_I; i++) { if (base + i < n) out[base + i] = run; run += v[i]; }
}

// bytes [w0, w1) of the output into out[0 .. w1 - w0): one warp per record, records from the last one that starts at or before w0
__global__ void __launch_bounds__(32 * VCF_WARPS) k_vcf_write(const VcfRec *rec, uint64_t n, const uint32_t *lists, const uint8_t *gt, const int32_t *gq,
                                                              const uint8_t *text, const unsigned long long *misc, const uint64_t *off,
                                                              const uint32_t *len, uint64_t w0, uint64_t w1, uint8_t *out)
{
	__shared__ VcfPlan plan[VCF_WARPS];
	const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
	VcfPlan &p = plan[wid];
	uint64_t lo = 0, hi = n;                                        // first record with off > w0, minus one
	while (lo < hi) { const uint64_t mid = (lo + hi) / 2; if (off[mid] <= w0) lo = mid + 1; else hi = mid; }
	const uint64_t r0 = lo ? lo - 1 : 0;
	const uint64_t step = (uint64_t)gridDim.x * VCF_WARPS;
	const int32_t gi = (int32_t)(long long)misc[M_GI];
	for (uint64_t r = r0 + (uint64_t)blockIdx.x * VCF_WARPS + wid; r < n && off[r] < w1; r += step) {
		const uint32_t m = len[r];
		if (!m) continue;
		const uint64_t a = off[r], b = a + m;
		if (b <= w0) continue;
		const VcfRec x = rec[r];
		const uint8_t *line = text + x.off;
		const uint32_t j0 = (uint32_t)(a < w0 ? w0 - a : 0), j1 = (uint32_t)(b > w1 ? w1 - a : m);
		uint8_t *dst = out + (a - w0);
		if (x.len_flags & VCF_LIT) {
			for (uint32_t j = j0 + lane; j < j1; j += 32) dst[j] = line[j];
			continue;
		}
		if (lane == 0) {
			const int64_t s = vcf_site(lists, x.list, gt);
			vcf_plan<true>(line, x.len_flags & VCF_LEN_MASK, x.len_flags, gt[s], gq[s], gi, &p);
		}
		__syncwarp();
		uint32_t piece = 0;
		for (uint32_t j = j0 + lane; j < j1; j += 32) dst[j] = vcf_plan_byte(p, line, j, piece);
		__syncwarp();
	}
}

// one BGZF member per block of text: member b to slots + b * DF_MEMBER_MAX, its size to msize[b]
__global__ void __launch_bounds__(32) k_deflate(const uint8_t *text, uint64_t n, uint8_t *slots, uint32_t *sym, uint32_t *msize)
{
	__shared__ DeflateWarp s;
	const uint64_t a = (uint64_t)blockIdx.x * DF_BLOCK;
	const uint32_t len = (uint32_t)min((uint64_t)DF_BLOCK, n - a);
	const uint32_t m = deflate_member(text + a, len, slots + (uint64_t)blockIdx.x * DF_MEMBER_MAX, sym + (uint64_t)blockIdx.x * DF_BLOCK, s);
	if (threadIdx.x == 0) msize[blockIdx.x] = m;
}

// members packed back to back: one block per member, 16-byte loads from the slot (slots are 64 KiB aligned)
__global__ void __launch_bounds__(256) k_member_compact(const uint8_t *slots, const uint32_t *moff, const uint32_t *msize, uint8_t *out)
{
	const uint8_t *src = slots + (uint64_t)blockIdx.x * DF_MEMBER_MAX;
	uint8_t *dst = out + moff[blockIdx.x];
	const uint32_t m = msize[blockIdx.x];
	for (uint32_t i = threadIdx.x * 16; i < m; i += 256 * 16) {
		const uint4 v = *reinterpret_cast<const uint4 *>(src + i);
		const uint8_t *b = reinterpret_cast<const uint8_t *>(&v);
		const uint32_t k = min(16u, m - i);
#pragma unroll
		for (uint32_t t = 0; t < 16; t++) if (t < k) dst[i + t] = b[t];
	}
}

// ---- buffers: the round's text and the pinned pair at the first write; the compressor's (members, LZ77 symbols: 0.4 GB) at the
// first BGZF write only ----
static int vcf_round_buffers(vgb_ctx *c, int bgzf)
{
	VcfState &v = c->vcf;
	if (!v.d_round) VGB_CUDA(c, cudaMalloc((void **)&v.d_round, VCF_ROUND));
	if (!v.d_misc) VGB_CUDA(c, cudaMalloc((void **)&v.d_misc, 8 * sizeof(unsigned long long)));
	if (!v.h_misc) VGB_CUDA(c, cudaMallocHost((void **)&v.h_misc, 8 * sizeof(unsigned long long)));
	for (int i = 0; i < 2; i++) {
		if (!v.h_out[i]) VGB_CUDA(c, cudaMallocHost((void **)&v.h_out[i], std::max(VCF_ROUND, VCF_OUT_CAP)));
		if (!v.ev[i]) VGB_CUDA(c, cudaEventCreateWithFlags(&v.ev[i], cudaEventDisableTiming));
	}
	if (bgzf) {
		if (!v.d_sym) VGB_CUDA(c, cudaMalloc((void **)&v.d_sym, (uint64_t)VCF_BLOCKS * DF_BLOCK * sizeof(uint32_t)));
		if (!v.d_packed) VGB_CUDA(c, cudaMalloc((void **)&v.d_packed, VCF_OUT_CAP));
		if (!v.d_msize) VGB_CUDA(c, cudaMalloc((void **)&v.d_msize, 2 * (VCF_BLOCKS + 1) * sizeof(uint32_t) + 64 * sizeof(uint32_t)));
		if (!v.d_slots) VGB_CUDA(c, cudaMalloc((void **)&v.d_slots, VCF_OUT_CAP));
	}
	return VGB_OK;
}

void vcf_free(vgb_ctx *c)
{
	VcfState &v = c->vcf;
	cudaFree(v.d_text); cudaFree(v.d_rec); cudaFree(v.d_lists); cudaFree(v.d_gt); cudaFree(v.d_gq); cudaFree(v.d_len); cudaFree(v.d_off);
	cudaFree(v.d_scan); cudaFree(v.d_round); cudaFree(v.d_slots); cudaFree(v.d_sym); cudaFree(v.d_packed); cudaFree(v.d_msize); cudaFree(v.d_misc);
	if (v.h_misc) cudaFreeHost(v.h_misc);
	for (int i = 0; i < 2; i++) {
		if (v.h_out[i]) cudaFreeHost(v.h_out[i]);
		if (v.ev[i]) cudaEventDestroy(v.ev[i]);
	}
	v = VcfState();
}

static void vcf_drop_template(VcfState &v)
{
	cudaFree(v.d_text); cudaFree(v.d_rec); cudaFree(v.d_lists); cudaFree(v.d_len); cudaFree(v.d_off); cudaFree(v.d_scan);
	v.d_text = nullptr; v.d_rec = nullptr; v.d_lists = nullptr; v.d_len = nullptr; v.d_off = nullptr; v.d_scan = nullptr;
	v.text_n = v.n_rec = v.n_lists = 0;
}

static int vcf_alloc_template(vgb_ctx *c, uint64_t text_n, uint64_t n_rec, uint64_t n_lists)
{
	VcfState &v = c->vcf;
	vcf_drop_template(v);
	VGB_CUDA(c, cudaMalloc((void **)&v.d_text, text_n ? text_n : 1));
	VGB_CUDA(c, cudaMalloc((void **)&v.d_rec, (n_rec ? n_rec : 1) * sizeof(VcfRec)));
	VGB_CUDA(c, cudaMalloc((void **)&v.d_lists, (n_lists ? n_lists : 1) * sizeof(uint32_t)));
	VGB_CUDA(c, cudaMalloc((void **)&v.d_len, (n_rec + 1) * sizeof(uint32_t)));
	VGB_CUDA(c, cudaMalloc((void **)&v.d_off, (n_rec + 1) * sizeof(uint64_t)));
	VGB_CUDA(c, cudaMalloc((void **)&v.d_scan, (n_rec / S64_TILE + 2) * sizeof(uint64_t)));
	v.text_n = text_n; v.n_rec = n_rec; v.n_lists = n_lists;
	return VGB_OK;
}

int vcf_template(vgb_ctx *c, const char *vcf, uint64_t n, const char *const *names, const uint64_t *lens, uint32_t n_contigs)
{
	if (!c->have_index) return set_err(c, VGB_E_ARG, "vgb_vcf_template needs the index (the sites) first");
	if (!vcf && n) return set_err(c, VGB_E_ARG, "vgb_vcf_template: no VCF bytes");
	const uint64_t n_sites = c->ix.n_sites;
	std::vector<uint32_t> pos(n_sites);
	if (n_sites) VGB_CUDA(c, copy_sync(c, pos.data(), c->d_site_pos, n_sites * sizeof(uint32_t), cudaMemcpyDeviceToHost));
	std::vector<std::string> nm;
	for (uint32_t j = 0; j < n_contigs; j++) nm.emplace_back(names[j] ? names[j] : "");
	std::vector<uint64_t> ln(lens, lens + n_contigs);
	VcfTemplate t;
	std::string err;
	if (!vcf_template_parse(vcf, n, nm, ln, pos.data(), n_sites, t, err)) return set_err(c, VGB_E_FORMAT, "%s", err.c_str());
	const uint64_t text_n = n + t.extra.size();
	if (text_n > (1ull << 40)) return set_err(c, VGB_E_ARG, "the VCF is larger than 1 TiB");
	int rc = vcf_alloc_template(c, text_n, t.rec.size(), t.lists.size());
	if (rc) return rc;
	VcfState &v = c->vcf;
	if (n) VGB_CUDA(c, copy_sync(c, v.d_text, vcf, n, cudaMemcpyHostToDevice));
	if (!t.extra.empty()) VGB_CUDA(c, copy_sync(c, v.d_text + n, t.extra.data(), t.extra.size(), cudaMemcpyHostToDevice));
	if (!t.rec.empty()) VGB_CUDA(c, copy_sync(c, v.d_rec, t.rec.data(), t.rec.size() * sizeof(VcfRec), cudaMemcpyHostToDevice));
	if (!t.lists.empty()) VGB_CUDA(c, copy_sync(c, v.d_lists, t.lists.data(), t.lists.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
	v.n_sites = n_sites;
	v.ready = true;
	return VGB_OK;
}

int vcf_template_copy(vgb_ctx *dst, vgb_ctx *src)
{
	if (!src->vcf.ready) return set_err(dst, VGB_E_ARG, "vgb_vcf_template_copy: the source context has no VCF template");
	if (!dst->have_index || dst->ix.n_sites != src->vcf.n_sites) return set_err(dst, VGB_E_ARG, "vgb_vcf_template_copy: the two contexts hold different indexes");
	const VcfState &s = src->vcf;
	int rc = vcf_alloc_template(dst, s.text_n, s.n_rec, s.n_lists);
	if (rc) return rc;
	VcfState &v = dst->vcf;
	VGB_CUDA(dst, cudaMemcpyPeerAsync(v.d_text, dst->device, s.d_text, src->device, s.text_n, dst->stream));
	VGB_CUDA(dst, cudaMemcpyPeerAsync(v.d_rec, dst->device, s.d_rec, src->device, s.n_rec * sizeof(VcfRec), dst->stream));
	VGB_CUDA(dst, cudaMemcpyPeerAsync(v.d_lists, dst->device, s.d_lists, src->device, s.n_lists * sizeof(uint32_t), dst->stream));
	VGB_CUDA(dst, cudaStreamSynchronize(dst->stream));
	v.n_sites = s.n_sites;
	v.ready = true;
	return VGB_OK;
}

// Rounds: text_round(k, dst) makes round k's bytes in dst (device), returns their count; with bgzf they are compressed.  Round k's
// bytes reach fn while round k + 1 is made.
template <typename F>
static int vcf_rounds(vgb_ctx *c, uint64_t total, int bgzf, int eof, vgb_write_fn fn, void *user, F text_round)
{
	VcfState &v = c->vcf;
	cudaStream_t st = c->stream;
	const uint64_t n_round = (total + VCF_ROUND - 1) / VCF_ROUND;
	uint64_t pending = 0;                                       // bytes of round k - 1 in h_out[(k - 1) & 1]
	for (uint64_t k = 0; k <= n_round; k++) {
		uint64_t bytes = 0;
		if (k < n_round) {
			const uint64_t w0 = k * VCF_ROUND, n = std::min(VCF_ROUND, total - w0);
			int rc = text_round(w0, n, v.d_round);
			if (rc) return rc;
			const uint8_t *res = v.d_round;
			if (bgzf) {
				const uint32_t nb = (uint32_t)((n + DF_BLOCK - 1) / DF_BLOCK);
				uint32_t *msize = v.d_msize, *moff = v.d_msize + VCF_BLOCKS + 1, *tmp = v.d_msize + 2 * (VCF_BLOCKS + 1);
				k_deflate<<<nb, 32, 0, st>>>(v.d_round, n, v.d_slots, v.d_sym, msize);
				if ((rc = exclusive_scan_u32(c, msize, moff, nb, tmp, moff + nb))) return rc;
				k_member_compact<<<nb, 256, 0, st>>>(v.d_slots, moff, msize, v.d_packed);
				c->launches += 2;
				VGB_CUDA(c, cudaGetLastError());
				VGB_CUDA(c, cudaMemcpyAsync(v.h_misc + M_OUT, moff + nb, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
				res = v.d_packed;
			}
			// round k - 1 to the caller while the device works on round k
			if (k > 0) {
				VGB_CUDA(c, cudaEventSynchronize(v.ev[(k - 1) & 1]));
				if (pending && fn(user, v.h_out[(k - 1) & 1], pending) != 0) return set_err(c, VGB_E_ARG, "the output callback failed");
				pending = 0;
			}
			VGB_CUDA(c, cudaStreamSynchronize(st));
			bytes = bgzf ? (uint64_t)*reinterpret_cast<const uint32_t *>(v.h_misc + M_OUT) : n;
			VGB_CUDA(c, cudaMemcpyAsync(v.h_out[k & 1], res, bytes, cudaMemcpyDeviceToHost, st));
			VGB_CUDA(c, cudaEventRecord(v.ev[k & 1], st));
			pending = bytes;
		} else if (k > 0) {
			VGB_CUDA(c, cudaEventSynchronize(v.ev[(k - 1) & 1]));
			if (pending && fn(user, v.h_out[(k - 1) & 1], pending) != 0) return set_err(c, VGB_E_ARG, "the output callback failed");
		}
	}
	if (bgzf && eof && fn(user, DF_EOF, sizeof(DF_EOF)) != 0) return set_err(c, VGB_E_ARG, "the output callback failed");
	return VGB_OK;
}

int vcf_write(vgb_ctx *c, const uint8_t *gt, const int32_t *gq, uint64_t n_sites, int bgzf, vgb_write_fn fn, void *user, uint64_t *text_bytes)
{
	VcfState &v = c->vcf;
	if (!v.ready) return set_err(c, VGB_E_ARG, "vgb_vcf_write: no VCF template (vgb_vcf_template)");
	if (n_sites != v.n_sites) return set_err(c, VGB_E_ARG, "vgb_vcf_write: %llu sites given, the index has %llu", (unsigned long long)n_sites,
	                                         (unsigned long long)v.n_sites);
	if (!fn || (n_sites && (!gt || !gq))) return set_err(c, VGB_E_ARG, "vgb_vcf_write: missing argument");
	int rc = vcf_round_buffers(c, bgzf);
	if (rc) return rc;
	cudaStream_t st = c->stream;
	if (v.site_cap < n_sites || !v.d_gt) {
		cudaFree(v.d_gt); cudaFree(v.d_gq);
		v.d_gt = nullptr; v.d_gq = nullptr;
		VGB_CUDA(c, cudaMalloc((void **)&v.d_gt, n_sites ? n_sites : 1));
		VGB_CUDA(c, cudaMalloc((void **)&v.d_gq, (n_sites ? n_sites : 1) * sizeof(int32_t)));
		v.site_cap = n_sites;
	}
	VGB_CUDA(c, cudaMemcpyAsync(v.d_gt, gt, n_sites, cudaMemcpyHostToDevice, st));
	VGB_CUDA(c, cudaMemcpyAsync(v.d_gq, gq, n_sites * sizeof(int32_t), cudaMemcpyHostToDevice, st));
	v.h_misc[M_ERR] = ~0ull; v.h_misc[M_FIRST] = ~0ull; v.h_misc[M_GI] = 0; v.h_misc[M_TOTAL] = 0;
	VGB_CUDA(c, cudaMemcpyAsync(v.d_misc, v.h_misc, 4 * sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
	const uint64_t n = v.n_rec;
	const unsigned g = (unsigned)((n + 255) / 256);
	if (n) {
		k_vcf_first<<<g, 256, 0, st>>>(v.d_rec, n, v.d_lists, v.d_gt, v.d_misc);
		k_vcf_gi<<<1, 1, 0, st>>>(v.d_rec, v.d_text, v.d_misc);
		k_vcf_size<<<g, 256, 0, st>>>(v.d_rec, n, v.d_lists, v.d_gt, v.d_gq, v.d_text, v.d_misc, v.d_len);
		c->launches += 3;
		VGB_CUDA(c, cudaGetLastError());
	}
	VGB_CUDA(c, cudaMemcpyAsync(v.h_misc, v.d_misc, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
	VGB_CUDA(c, cudaStreamSynchronize(st));
	if (v.h_misc[M_ERR] != ~0ull) return set_err(c, VGB_E_FORMAT, "%s", vcf_error_text((int)(v.h_misc[M_ERR] & 7)));
	const uint64_t total = v.h_misc[M_TOTAL];
	if (n) {
		const uint64_t nt = (n + S64_TILE - 1) / S64_TILE;
		k_scan64_tiles<<<(unsigned)nt, S64_T, 0, st>>>(v.d_len, n, v.d_scan);
		k_scan64_top<<<1, 1024, 0, st>>>(v.d_scan, nt);
		k_scan64_apply<<<(unsigned)nt, S64_T, 0, st>>>(v.d_len, n, v.d_scan, v.d_off);
		c->launches += 3;
		VGB_CUDA(c, cudaGetLastError());
	}
	if (text_bytes) *text_bytes = total;
	const unsigned wg = (unsigned)std::min<uint64_t>((n + VCF_WARPS - 1) / VCF_WARPS, (uint64_t)c->sm_count * 16);
	return vcf_rounds(c, total, bgzf, 1, fn, user, [&](uint64_t w0, uint64_t bytes, uint8_t *dst) -> int {
		k_vcf_write<<<wg ? wg : 1, 32 * VCF_WARPS, 0, st>>>(v.d_rec, n, v.d_lists, v.d_gt, v.d_gq, v.d_text, v.d_misc, v.d_off, v.d_len, w0,
		                                                  w0 + bytes, dst);
		c->launches++;
		VGB_CUDA(c, cudaGetLastError());
		return VGB_OK;
	});
}

int deflate_bgzf(vgb_ctx *c, const void *text, uint64_t nbytes, int on_device, int eof, vgb_write_fn fn, void *user)
{
	if (!fn || (!text && nbytes)) return set_err(c, VGB_E_ARG, "vgb_deflate_bgzf: missing argument");
	int rc = vcf_round_buffers(c, 1);
	if (rc) return rc;
	const uint8_t *p = static_cast<const uint8_t *>(text);
	return vcf_rounds(c, nbytes, 1, eof, fn, user, [&](uint64_t w0, uint64_t bytes, uint8_t *dst) -> int {
		VGB_CUDA(c, cudaMemcpyAsync(dst, p + w0, bytes, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream));
		return VGB_OK;
	});
}

}  // namespace vgb
