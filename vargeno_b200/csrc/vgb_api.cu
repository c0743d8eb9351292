// vgb_api.cu -- the C ABI (include/vgb200.h): context, chunk pipeline, statistics.
#include <cstdarg>
#include <algorithm>
#include <cstring>
#include <vector>

#include "vgb_internal.h"

namespace vgb {

thread_local std::string g_create_err;

int set_err(vgb_ctx *c, int code, const char *fmt, ...)
{
	char buf[1024];
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(buf, sizeof(buf), fmt, ap);
	va_end(ap);
	if (c) c->err = buf; else g_create_err = buf;
	return code;
}

}  // namespace vgb

using namespace vgb;

extern "C" {

int vgb_abi_version(void) { return VGB_ABI_VERSION; }

const char *vgb_last_error(const vgb_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int vgb_nccl_unique_id(void *out128)
{
	std::string err;
	const int rc = nccl_unique_id(out128, err);
	if (rc) g_create_err = err;
	return rc;
}

int vgb_ctx_create(vgb_ctx **out, const vgb_config *cfg)
{
	if (!out || !cfg) return set_err(nullptr, VGB_E_ARG, "null argument");
	*out = nullptr;
	int ndev = 0;
	cudaError_t e = cudaGetDeviceCount(&ndev);
	if (e != cudaSuccess || ndev == 0)
		return set_err(nullptr, VGB_E_CUDA, "no CUDA device (%s): libvgb200 has no CPU fallback", e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
	if (cfg->device < 0 || cfg->device >= ndev) return set_err(nullptr, VGB_E_ARG, "device %d out of range (%d devices)", cfg->device, ndev);
	if (cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size) return set_err(nullptr, VGB_E_ARG, "bad world_size / rank");
	if (cfg->world_size > 1 && !cfg->nccl_unique_id) return set_err(nullptr, VGB_E_ARG, "world_size > 1 needs an NCCL unique id");
	cudaDeviceProp prop;
	if ((e = cudaSetDevice(cfg->device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, cfg->device)) != cudaSuccess)
		return set_err(nullptr, VGB_E_CUDA, "cudaSetDevice(%d): %s", cfg->device, cudaGetErrorString(e));
	if (prop.major < 10) return set_err(nullptr, VGB_E_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", cfg->device, prop.major, prop.minor);

	vgb_ctx *c = new vgb_ctx();
	c->cfg = *cfg;
	c->device = cfg->device;
	c->sm_count = prop.multiProcessorCount;
	c->max_chunk_bytes = cfg->max_chunk_bytes ? cfg->max_chunk_bytes : (256ull << 20);
	if (c->max_chunk_bytes > 0xFFFFFF00ull) { delete c; return set_err(nullptr, VGB_E_ARG, "max_chunk_bytes must stay below 4 GiB (32-bit line offsets)"); }
	c->max_chunk_bytes = (c->max_chunk_bytes + 4095) & ~4095ull;
#define CK(call) do { if ((e = (call)) != cudaSuccess) { set_err(nullptr, VGB_E_CUDA, "%s: %s", #call, cudaGetErrorString(e)); vgb_ctx_destroy(c); return VGB_E_CUDA; } } while (0)
	CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
	CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
	CK(cudaStreamCreateWithFlags(&c->tail_stream, cudaStreamNonBlocking));

	for (int i = 0; i < 4; i++) CK(cudaEventCreate(&c->ev[i]));
	CK(cudaMalloc((void **)&c->d_stats, sizeof(DevStats)));
	CK(vgb::memset_sync(c, c->d_stats, 0, sizeof(DevStats)));
	CK(cudaMalloc((void **)&c->d_tables, (64 * 64 * 3 + 127) * sizeof(double)));
	{
		std::vector<double> t(64 * 64 * 3 + 127);
		build_call_tables(t.data(), t.data() + 64 * 64 * 3);
		CK(vgb::copy_sync(c, c->d_tables, t.data(), t.size() * sizeof(double), cudaMemcpyHostToDevice));
	}
	const uint64_t nblk = c->max_chunk_bytes / 4096 + 2;
	for (int s = 0; s < 2; s++) {
		Chunk &k = c->chunk[s];
		CK(cudaMalloc((void **)&k.d_text, c->max_chunk_bytes + 64));
		CK(cudaMalloc((void **)&k.d_line_start, (c->max_chunk_bytes / 2 + 16) * 4));
		CK(cudaMalloc((void **)&k.d_blk_counts, (2 * nblk + 64) * 4));
		CK(cudaMalloc((void **)&k.d_defer, (c->max_chunk_bytes / 8 + 16) * 4));
		CK(cudaMalloc((void **)&k.d_defer2, (c->max_chunk_bytes / 8 + 16) * 4));
		CK(cudaMalloc((void **)&k.d_defer3, (c->max_chunk_bytes / 8 + 16) * 4));
		CK(cudaMalloc((void **)&k.d_meta, 64));
		CK(vgb::memset_sync(c, k.d_meta, 0, 64));
		CK(cudaEventCreateWithFlags(&k.copied, cudaEventDisableTiming));
		CK(cudaEventCreate(&k.done));
		CK(cudaEventCreate(&k.t0));
		CK(cudaEventCreate(&k.t1));
		CK(cudaEventCreate(&k.g0));
		CK(cudaEventCreate(&k.g1));
		CK(cudaEventCreate(&k.h0));
	}
#undef CK
	if (cfg->world_size > 1) {
		const int rc = nccl_init(c);
		if (rc) { g_create_err = c->err; vgb_ctx_destroy(c); return rc; }
	}
	*out = c;
	return VGB_OK;
}

int vgb_comm_init(vgb_ctx *c, int32_t world_size, int32_t rank, const void *uid)
{
	if (!c) return VGB_E_ARG;
	if (world_size < 2 || rank < 0 || rank >= world_size || !uid) return set_err(c, VGB_E_ARG, "bad world_size / rank / unique id");
	if (c->nccl_comm || c->cfg.world_size != 1) return set_err(c, VGB_E_ARG, "context already belongs to a communicator");
	cudaSetDevice(c->device);
	memcpy(c->uid, uid, 128);
	c->cfg.world_size = world_size; c->cfg.rank = rank; c->cfg.nccl_unique_id = c->uid;
	const int rc = nccl_init(c);
	if (rc) { c->cfg.world_size = 1; c->cfg.rank = 0; c->cfg.nccl_unique_id = nullptr; }
	return rc;
}

void vgb_ctx_destroy(vgb_ctx *c)
{
	if (!c) return;
	cudaSetDevice(c->device);
	cudaDeviceSynchronize();
	nccl_destroy(c);
	for (int i = 0; i < c->n_owned; i++) cudaFree(c->owned[i]);
	for (int s = 0; s < 2; s++) {
		Chunk &k = c->chunk[s];
		cudaFree(k.d_text); cudaFree(k.d_line_start); cudaFree(k.d_blk_counts); cudaFree(k.d_meta); cudaFree(k.d_defer); cudaFree(k.d_defer2); cudaFree(k.d_defer3);
		cudaFree(k.d_comp); cudaFree(k.d_blk);
		if (k.h_blk) cudaFreeHost(k.h_blk);
		if (k.h_pinned) cudaFreeHost(k.h_pinned);
		if (k.copied) cudaEventDestroy(k.copied);
		if (k.done) cudaEventDestroy(k.done);
		if (k.t0) cudaEventDestroy(k.t0);
		if (k.t1) cudaEventDestroy(k.t1);
		if (k.g0) cudaEventDestroy(k.g0);
		if (k.g1) cudaEventDestroy(k.g1);
		if (k.h0) cudaEventDestroy(k.h0);
	}
	gzip_free(c);
	bam_free(c);
	vcf_free(c);
	cudaFree(c->d_stats); cudaFree(c->d_tables); cudaFree(c->d_trace);
	for (int i = 0; i < 4; i++) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
	if (c->stream) cudaStreamDestroy(c->stream);
	if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
	if (c->tail_stream) cudaStreamDestroy(c->tail_stream);
	delete c;
}

int vgb_index_upload(vgb_ctx *c, const vgb_index_view *view)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return index_upload(c, view);
}

int vgb_site_count(vgb_ctx *c, uint64_t *n)
{
	if (!c || !n) return VGB_E_ARG;
	if (!c->have_index) return set_err(c, VGB_E_ARG, "no index");
	*n = c->ix.n_sites;
	return VGB_OK;
}

int vgb_fetch_sites(vgb_ctx *c, uint32_t *pos, uint8_t *code, uint8_t *rf, uint8_t *af, uint64_t n)
{
	if (!c) return VGB_E_ARG;
	if (!c->have_index) return set_err(c, VGB_E_ARG, "no index");
	if (n != c->ix.n_sites) return set_err(c, VGB_E_ARG, "n_sites mismatch");
	cudaSetDevice(c->device);
	if (n == 0) return VGB_OK;
	if (pos) VGB_CUDA(c, vgb::copy_sync(c, pos, c->d_site_pos, n * 4, cudaMemcpyDeviceToHost));
	if (code) VGB_CUDA(c, vgb::copy_sync(c, code, c->ix.site_code, n, cudaMemcpyDeviceToHost));
	if (rf) VGB_CUDA(c, vgb::copy_sync(c, rf, c->d_site_rf, n, cudaMemcpyDeviceToHost));
	if (af) VGB_CUDA(c, vgb::copy_sync(c, af, c->d_site_af, n, cudaMemcpyDeviceToHost));
	return VGB_OK;
}

int vgb_pinned_buffer(vgb_ctx *c, int slot, char **ptr, uint64_t *cap)
{
	if (!c || slot < 0 || slot > 1 || !ptr) return VGB_E_ARG;
	cudaSetDevice(c->device);
	Chunk &k = c->chunk[slot];
	if (!k.h_pinned) VGB_CUDA(c, cudaMallocHost((void **)&k.h_pinned, c->max_chunk_bytes));
	VGB_CUDA(c, cudaEventSynchronize(k.copied));       // the H2D copy out of this buffer has finished
	*ptr = k.h_pinned;
	if (cap) *cap = c->max_chunk_bytes;
	return VGB_OK;
}

}  // extern "C"

namespace vgb {

void collect_times(vgb_ctx *c, int slot)
{
	Chunk &k = c->chunk[slot];
	if (!k.busy) return;
	cudaEventSynchronize(k.done);
	float a = 0, b = 0;
	if (cudaEventElapsedTime(&a, k.t0, k.t1) == cudaSuccess) c->ms_parse += a;
	if (k.tail) {
		// main kernels on the kernel stream + hand-over kernels on the tail stream (which ran under the next chunk's kernels:
		// both intervals include what the overlap costs them)
		float t = 0;
		if (cudaEventElapsedTime(&b, k.g0, k.g1) == cudaSuccess) c->ms_geno += b;
		if (cudaEventElapsedTime(&t, k.h0, k.done) == cudaSuccess) c->ms_geno += t;
	} else if (cudaEventElapsedTime(&b, k.g0, k.done) == cudaSuccess) c->ms_geno += b;
	k.busy = false;
}

// the text of the chunk is (or will be, in stream order) in k.d_text: record framing, then the per-read kernels
int process_text(vgb_ctx *c, Chunk &k, uint64_t nbytes, uint64_t first_read_id, int window, uint64_t ov, int last)
{
	k.tail = false;
	if (!window) VGB_CUDA(c, cudaEventRecord(k.t0, c->stream));      // BGZF chunks: recorded in front of the inflate kernel, which counts as parsing
	int rc = fastq_index_lines(c, k, nbytes, c->stream, window, ov, last);
	if (rc == VGB_OK) {
		VGB_CUDA(c, cudaEventRecord(k.t1, c->stream));
		if (c->cfg.flags & VGB_CFG_TRACE) {
			// the trace is indexed by read ordinal: learn this chunk's read count and grow the buffer
			uint32_t meta[4];
			VGB_CUDA(c, cudaMemcpyAsync(meta, k.d_meta, 16, cudaMemcpyDeviceToHost, c->stream));
			VGB_CUDA(c, cudaStreamSynchronize(c->stream));
			const uint64_t need = c->trace_n + meta[1];
			if (need > c->trace_cap) {
				const uint64_t cap = std::max<uint64_t>(need, c->trace_cap * 2 + 1024);
				vgb_read_result *nt = nullptr;
				VGB_CUDA(c, cudaStreamSynchronize(c->stream));       // earlier chunks still write the old buffer
				VGB_CUDA(c, cudaMalloc((void **)&nt, cap * sizeof(vgb_read_result)));
				if (c->trace_n) VGB_CUDA(c, vgb::copy_sync(c, nt, c->d_trace, c->trace_n * sizeof(vgb_read_result), cudaMemcpyDeviceToDevice));
				cudaFree(c->d_trace);
				c->d_trace = nt; c->trace_cap = cap;
			}
			VGB_CUDA(c, cudaEventRecord(k.g0, c->stream));
			rc = geno_launch(c, k, nbytes, first_read_id);
			c->trace_n = need;
		} else {
			VGB_CUDA(c, cudaEventRecord(k.g0, c->stream));
			rc = geno_launch(c, k, nbytes, first_read_id);
		}
	}
	cudaEventRecord(k.done, k.tail ? c->tail_stream : c->stream);
	k.busy = true;
	c->chunks++;
	c->chunk_bytes += nbytes;
	return rc;
}

static int submit_common(vgb_ctx *c, const char *host_chunk, const char *device_chunk, uint64_t nbytes, uint64_t first_read_id)
{
	if (!c) return VGB_E_ARG;
	if (!c->have_index) return set_err(c, VGB_E_ARG, "vgb_index_upload has not been called");
	if (nbytes > c->max_chunk_bytes) return set_err(c, VGB_E_ARG, "chunk of %llu bytes exceeds max_chunk_bytes %llu", (unsigned long long)nbytes, (unsigned long long)c->max_chunk_bytes);
	if (nbytes == 0) return VGB_OK;
	cudaSetDevice(c->device);
	const int slot = c->next_slot;
	c->next_slot ^= 1;
	Chunk &k = c->chunk[slot];
	collect_times(c, slot);                            // waits until the previous chunk in this slot is done
	char *own_text = k.d_text;
	// Two streams: the H2D copy of chunk i+1 runs under the kernels of chunk i.  Record framing stays on the kernel stream:
	// k_geno8 is a persistent grid that fills every SM, so a framing kernel on a third stream only gets the SMs when k_geno8
	// drains (measured: 1.5 % on the step, and both kernels' event times stop meaning anything).
	if (device_chunk) {
		k.d_text = const_cast<char *>(device_chunk);   // resident input: no copy at all
	} else {
		VGB_CUDA(c, cudaMemcpyAsync(k.d_text, host_chunk, nbytes, cudaMemcpyHostToDevice, c->copy_stream));
		VGB_CUDA(c, cudaEventRecord(k.copied, c->copy_stream));
		VGB_CUDA(c, cudaStreamWaitEvent(c->stream, k.copied, 0));
		auto in_pinned = [&](const Chunk &q) { return q.h_pinned && host_chunk >= q.h_pinned && host_chunk < q.h_pinned + c->max_chunk_bytes; };
		if (!in_pinned(k) && !in_pinned(c->chunk[slot ^ 1]))
			VGB_CUDA(c, cudaEventSynchronize(k.copied));   // caller's own memory: safe to reuse on return
	}
	const int rc = process_text(c, k, nbytes, first_read_id, 0, 0, 0);
	if (device_chunk) k.d_text = own_text;
	return rc;
}

// the compressed members of a BGZF call into slot k's buffers (copy stream; the kernel stream waits for it) and their table; *out =
// the sum of their ISIZEs.  Called with the slot free (collect_times).
int bgzf_stage(vgb_ctx *c, Chunk &k, int slot, const uint8_t *comp, uint64_t comp_bytes, const vgb_bgzf_member *mem, uint32_t n_mem, uint64_t *out)
{
	*out = 0;
	if (n_mem == 0) return VGB_OK;
	if (!k.d_comp) VGB_CUDA(c, cudaMalloc((void **)&k.d_comp, c->max_chunk_bytes + 64));
	if (k.blk_cap < n_mem) {
		const uint32_t cap = std::max<uint32_t>(n_mem, 2 * k.blk_cap + 1024);
		if (k.d_blk) cudaFree(k.d_blk);
		if (k.h_blk) cudaFreeHost(k.h_blk);
		k.d_blk = nullptr; k.h_blk = nullptr; k.blk_cap = 0;
		VGB_CUDA(c, cudaMalloc((void **)&k.d_blk, (size_t)cap * sizeof(BgzfBlock)));
		VGB_CUDA(c, cudaMallocHost((void **)&k.h_blk, (size_t)cap * sizeof(BgzfBlock)));
		k.blk_cap = cap;
	}
	uint64_t o = 0;
	for (uint32_t i = 0; i < n_mem; i++) {
		if ((uint64_t)mem[i].comp_offset + mem[i].comp_len > comp_bytes || mem[i].out_len > 65536)
			return set_err(c, VGB_E_ARG, "BGZF member %u lies outside the chunk or claims more than 64 KiB", i);
		k.h_blk[i] = BgzfBlock{ mem[i].comp_offset, mem[i].comp_len, (uint32_t)o, mem[i].out_len };
		o += mem[i].out_len;
	}
	if (o > c->max_chunk_bytes) return set_err(c, VGB_E_ARG, "chunk inflates to %llu bytes, more than max_chunk_bytes", (unsigned long long)o);
	VGB_CUDA(c, cudaMemcpyAsync(k.d_comp, comp, comp_bytes, cudaMemcpyHostToDevice, c->copy_stream));
	VGB_CUDA(c, cudaMemcpyAsync(k.d_blk, k.h_blk, (size_t)n_mem * sizeof(BgzfBlock), cudaMemcpyHostToDevice, c->copy_stream));
	VGB_CUDA(c, cudaEventRecord(k.copied, c->copy_stream));
	VGB_CUDA(c, cudaStreamWaitEvent(c->stream, k.copied, 0));
	const char *hc = (const char *)comp;
	auto in_pinned = [&](const Chunk &q) { return q.h_pinned && hc >= q.h_pinned && hc < q.h_pinned + c->max_chunk_bytes; };
	if (!in_pinned(k) && !in_pinned(c->chunk[slot ^ 1])) VGB_CUDA(c, cudaEventSynchronize(k.copied));
	*out = o;
	return VGB_OK;
}

// BGZF chunk: compressed members over PCIe, inflated on the device straight into the chunk's text buffer
static int submit_bgzf(vgb_ctx *c, const uint8_t *comp, uint64_t comp_bytes, const vgb_bgzf_member *mem, uint32_t n_mem, uint64_t ov, int last)
{
	if (!c->have_index) return set_err(c, VGB_E_ARG, "vgb_index_upload has not been called");
	if (comp_bytes > c->max_chunk_bytes) return set_err(c, VGB_E_ARG, "compressed chunk of %llu bytes exceeds max_chunk_bytes", (unsigned long long)comp_bytes);
	if (n_mem == 0) return VGB_OK;
	cudaSetDevice(c->device);
	const int slot = c->next_slot;
	c->next_slot ^= 1;
	Chunk &k = c->chunk[slot];
	collect_times(c, slot);
	uint64_t out = 0;
	const int rs = bgzf_stage(c, k, slot, comp, comp_bytes, mem, n_mem, &out);
	if (rs != VGB_OK) return rs;
	if (ov > out) return set_err(c, VGB_E_ARG, "overlap larger than the chunk");
	if (out == 0) { cudaEventRecord(k.done, c->stream); k.busy = true; return VGB_OK; }
	VGB_CUDA(c, cudaEventRecord(k.t0, c->stream));
	int rc = bgzf_inflate(c, k, k.d_comp, k.d_blk, n_mem, c->stream, reinterpret_cast<uint8_t *>(k.d_text));
	if (rc != VGB_OK) return rc;
	return process_text(c, k, out, 0, 1, ov, last);
}

}  // namespace vgb

extern "C" {

int vgb_submit_fastq(vgb_ctx *c, const char *chunk, uint64_t nbytes, uint64_t first_read_id)
{
	if (!chunk && nbytes) return c ? set_err(c, VGB_E_ARG, "null chunk") : VGB_E_ARG;
	return submit_common(c, chunk, nullptr, nbytes, first_read_id);
}

int vgb_submit_fastq_device(vgb_ctx *c, const char *device_chunk, uint64_t nbytes, uint64_t first_read_id)
{
	if (!device_chunk && nbytes) return c ? set_err(c, VGB_E_ARG, "null chunk") : VGB_E_ARG;
	return submit_common(c, nullptr, device_chunk, nbytes, first_read_id);
}

int vgb_submit_bgzf(vgb_ctx *c, const void *comp, uint64_t comp_bytes, const vgb_bgzf_member *members, uint32_t n_members, uint64_t overlap_bytes, int last_chunk)
{
	if (!c || (n_members && (!comp || !members))) return c ? set_err(c, VGB_E_ARG, "null argument") : VGB_E_ARG;
	return submit_bgzf(c, (const uint8_t *)comp, comp_bytes, members, n_members, overlap_bytes, last_chunk);
}

int vgb_submit_gzip(vgb_ctx *c, const void *comp, uint64_t comp_bytes, int first, int last)
{
	if (!c || (comp_bytes && !comp)) return c ? set_err(c, VGB_E_ARG, "null argument") : VGB_E_ARG;
	return submit_gzip(c, (const uint8_t *)comp, comp_bytes, first, last);
}

int vgb_submit_bam(vgb_ctx *c, const void *comp, uint64_t comp_bytes, const vgb_bgzf_member *members, uint32_t n_members, int first, int last)
{
	if (!c || (n_members && (!comp || !members))) return c ? set_err(c, VGB_E_ARG, "null argument") : VGB_E_ARG;
	if (comp_bytes > c->max_chunk_bytes) return set_err(c, VGB_E_ARG, "compressed BAM piece of %llu bytes exceeds max_chunk_bytes", (unsigned long long)comp_bytes);
	return submit_bam(c, (const uint8_t *)comp, comp_bytes, members, n_members, first, last);
}

int vgb_sync(vgb_ctx *c)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	VGB_CUDA(c, cudaStreamSynchronize(c->tail_stream));
	VGB_CUDA(c, cudaStreamSynchronize(c->copy_stream));
	VGB_CUDA(c, cudaStreamSynchronize(c->stream));
	collect_times(c, 0);
	collect_times(c, 1);
	uint32_t bits = 0;
	for (int s = 0; s < 2; s++) {
		uint32_t meta[6] = { 0, 0, 0, 0, 0, 0 };
		VGB_CUDA(c, vgb::copy_sync(c, meta, c->chunk[s].d_meta, 24, cudaMemcpyDeviceToHost));
		bits |= meta[3] | meta[5];
	}
	DevStats st;
	VGB_CUDA(c, vgb::copy_sync(c, &st, c->d_stats, sizeof(st), cudaMemcpyDeviceToHost));
	c->sticky_format |= bits;
	if (c->sticky_format & 8) return set_err(c, VGB_E_FORMAT, "BGZF input: a gzip member is corrupt or does not inflate to the size its trailer states");
	if (c->sticky_format & 16) return set_err(c, VGB_E_FORMAT, "gzip input: %s", c->gz.err.c_str());
	if (c->sticky_format & 32)
		return set_err(c, VGB_E_FORMAT, "BAM input: %s (%llu records with more than 1022 bases)", c->bam.err.c_str(), (unsigned long long)c->bam.long_records);
	if (c->sticky_format || st.bad_records)
		return set_err(c, VGB_E_FORMAT, "FASTQ input violates the contract:%s%s%s (%llu bad records)",
		               (c->sticky_format & 1) ? " truncated record (line count not a multiple of 4);" : "",
		               (c->sticky_format & 2) ? " line longer than 1022 characters, base outside ACGTNacgtn or quality line too short;" : "",
		               (c->sticky_format & 4) ? " too many lines for max_chunk_bytes;" : "", st.bad_records);
	if (st.overflow_reads)
		return set_err(c, VGB_E_OVERFLOW, "%llu reads produced more than 2000 hit contexts per dictionary (the reference overflows its arrays, src/qv.cc:709,728-729)", st.overflow_reads);
	if (st.freq_wrap_reads)
		return set_err(c, VGB_E_OVERFLOW, "%llu reads gave one position more than 255 votes (the reference's uint8 vote counter wraps there, src/qv.cc:57-93; results for these reads would differ)", st.freq_wrap_reads);
	return VGB_OK;
}

int vgb_reset_counts(vgb_ctx *c)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	VGB_CUDA(c, cudaStreamSynchronize(c->tail_stream));
	VGB_CUDA(c, cudaStreamSynchronize(c->copy_stream));
	VGB_CUDA(c, cudaStreamSynchronize(c->stream));
	VGB_CUDA(c, vgb::memset_sync(c, c->d_stats, 0, sizeof(DevStats)));
	if (c->have_index && c->ix.n_sites) VGB_CUDA(c, vgb::memset_sync(c, c->ix.cnt, 0, 2 * c->ix.n_sites * 4));
	for (int s = 0; s < 2; s++) VGB_CUDA(c, vgb::memset_sync(c, c->chunk[s].d_meta, 0, 64));
	c->trace_n = 0; c->sticky_format = 0;
	c->chunks = c->chunk_bytes = 0; c->ms_parse = c->ms_geno = 0; c->launches = 0;
	if (c->have_index && getenv("VGB_RETUNE")) return geno_prepare(c);   // tuning runs: re-read the VGB_* kernel knobs without a new index upload
	return VGB_OK;
}

int vgb_reset_sample(vgb_ctx *c)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	VGB_CUDA(c, cudaStreamSynchronize(c->tail_stream));
	VGB_CUDA(c, cudaStreamSynchronize(c->copy_stream));
	VGB_CUDA(c, cudaStreamSynchronize(c->stream));
	collect_times(c, 0);                                     // the last chunks' event times belong to the sample that ends here
	collect_times(c, 1);
	const int rc = vgb_reset_counts(c);
	if (rc != VGB_OK) return rc;
	gzip_reset(c);
	bam_reset(c);
	return VGB_OK;
}

int vgb_vcf_template(vgb_ctx *c, const char *vcf, uint64_t nbytes, const char *const *contig_names, const uint64_t *contig_lens, uint32_t n_contigs)
{
	if (!c || (n_contigs && (!contig_names || !contig_lens))) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return vcf_template(c, vcf, nbytes, contig_names, contig_lens, n_contigs);
}

int vgb_vcf_template_copy(vgb_ctx *dst, vgb_ctx *src)
{
	if (!dst || !src) return VGB_E_ARG;
	cudaSetDevice(dst->device);
	return vcf_template_copy(dst, src);
}

int vgb_vcf_write(vgb_ctx *c, const uint8_t *gtype, const int32_t *gq, uint64_t n_sites, int bgzf, vgb_write_fn fn, void *user, uint64_t *text_bytes)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return vcf_write(c, gtype, gq, n_sites, bgzf, fn, user, text_bytes);
}

int vgb_deflate_bgzf(vgb_ctx *c, const void *text, uint64_t nbytes, int text_on_device, int eof, vgb_write_fn fn, void *user)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return deflate_bgzf(c, text, nbytes, text_on_device, eof, fn, user);
}

int vgb_fetch_read_results(vgb_ctx *c, vgb_read_result *out, uint64_t cap, uint64_t *n)
{
	if (!c || !n) return VGB_E_ARG;
	if (!(c->cfg.flags & VGB_CFG_TRACE)) return set_err(c, VGB_E_ARG, "context was created without VGB_CFG_TRACE");
	cudaSetDevice(c->device);
	VGB_CUDA(c, cudaStreamSynchronize(c->stream));
	*n = c->trace_n;
	const uint64_t m = std::min(cap, c->trace_n);
	if (out && m) VGB_CUDA(c, vgb::copy_sync(c, out, c->d_trace, m * sizeof(vgb_read_result), cudaMemcpyDeviceToHost));
	return VGB_OK;
}

int vgb_lookup_kmers(vgb_ctx *c, const uint64_t *kmers, uint64_t n, vgb_hit *out)
{
	if (!c || (n && (!kmers || !out))) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return lookup_kmers(c, kmers, n, out);
}

int vgb_allreduce_pileup(vgb_ctx *c)
{
	if (!c) return VGB_E_ARG;
	if (!c->have_index) return set_err(c, VGB_E_ARG, "no index");
	if (c->cfg.world_size == 1) return VGB_OK;
	cudaSetDevice(c->device);
	VGB_CUDA(c, cudaStreamSynchronize(c->tail_stream));      // the hand-over kernels of the last chunks update the counters too
	const int rc = nccl_allreduce_u32(c, c->ix.cnt, 2 * c->ix.n_sites);
	if (rc) return rc;
	VGB_CUDA(c, cudaStreamSynchronize(c->stream));
	return VGB_OK;
}

int vgb_fetch_pileup(vgb_ctx *c, uint32_t *ref_cnt, uint32_t *alt_cnt, uint64_t n_sites)
{
	if (!c || (n_sites && (!ref_cnt || !alt_cnt))) return VGB_E_ARG;
	cudaSetDevice(c->device);
	VGB_CUDA(c, cudaStreamSynchronize(c->tail_stream));      // the hand-over kernels of the last chunks update the counters too
	return fetch_pileup(c, ref_cnt, alt_cnt, n_sites);
}

int vgb_call(vgb_ctx *c, uint8_t *gtype, double *conf, uint64_t n_sites)
{
	if (!c || (n_sites && (!gtype || !conf))) return VGB_E_ARG;
	cudaSetDevice(c->device);
	VGB_CUDA(c, cudaStreamSynchronize(c->tail_stream));      // the hand-over kernels of the last chunks update the counters too
	return call_sites(c, gtype, conf, n_sites);
}

int vgb_counter_device_ptr(vgb_ctx *c, void **ptr, uint64_t *n_u32)
{
	if (!c || !ptr || !n_u32) return VGB_E_ARG;
	if (!c->have_index) return set_err(c, VGB_E_ARG, "no index");
	*ptr = c->ix.cnt;
	*n_u32 = 2 * c->ix.n_sites;
	return VGB_OK;
}

int vgb_get_stats(vgb_ctx *c, vgb_stats *out)
{
	if (!c || !out) return VGB_E_ARG;
	cudaSetDevice(c->device);
	VGB_CUDA(c, cudaStreamSynchronize(c->tail_stream));      // the hand-over kernels of the last chunks update the counters too
	VGB_CUDA(c, cudaStreamSynchronize(c->stream));
	collect_times(c, 0);
	collect_times(c, 1);
	DevStats st;
	VGB_CUDA(c, vgb::copy_sync(c, &st, c->d_stats, sizeof(st), cudaMemcpyDeviceToHost));
	memset(out, 0, sizeof(*out));
	out->reads = st.reads; out->skipped_n = st.skipped_n; out->passes = st.passes; out->placed = st.placed;
	out->exact_lookups = st.exact_lookups; out->nbr_query_lookups = st.nbr_query_lookups; out->nbr_scan_reads = st.nbr_scan_reads;
	out->bf_probes = st.bf_probes; out->lowq_kmers = st.lowq_kmers; out->events = st.events; out->pileup_incr = st.pileup_incr;
	out->big_kmers = st.big_kmers; out->bad_records = st.bad_records;
	out->chunks = c->chunks; out->chunk_bytes = c->chunk_bytes;
	out->gpu_ms_parse = c->ms_parse; out->gpu_ms_geno = c->ms_geno; out->kernel_launches = c->launches;
	out->freq_wrap_reads = st.freq_wrap_reads;
	return VGB_OK;
}

int vgb_probe_bench(vgb_ctx *c, uint64_t n, int mode, uint64_t seed, int repeats, double *ms, uint64_t *found)
{
	if (!c || !ms || !found || n == 0) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return probe_bench(c, n, mode, seed, repeats, ms, found);
}

int vgb_random_sector_bench(vgb_ctx *c, uint64_t bytes, uint64_t n_loads, int repeats, double *gbs)
{
	if (!c || !gbs || bytes < 4096 || n_loads == 0) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return random_sector_bench(c, bytes, n_loads, repeats, gbs);
}

int vgb_synth_reads_device(vgb_ctx *c, const uint8_t *hap0, const uint8_t *hap1, uint64_t genome_len, const uint64_t *cstart,
                           const uint64_t *clen, uint32_t n_contigs, uint64_t n_reads, uint32_t read_len, uint64_t seed,
                           uint64_t first_id, uint32_t id_width, double sub_rate, double lowq_prob, uint32_t lowq_chars,
                           char *out, uint64_t out_cap)
{
	if (!c || !hap0 || !hap1 || !cstart || !clen || !out || n_contigs == 0) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return synth_reads(c, hap0, hap1, genome_len, cstart, clen, n_contigs, n_reads, read_len, seed, first_id, id_width, sub_rate,
	                   lowq_prob, lowq_chars, out, out_cap);
}

int vgb_build_index_device(vgb_ctx *c, const uint8_t *device_genome, uint64_t genome_len, const uint64_t *cstart, const uint64_t *clen,
                           uint32_t n_contigs, const uint32_t *snp_pos0, const uint8_t *snp_code, const uint8_t *snp_rf, const uint8_t *snp_af,
                           uint64_t n_snp_lines, const uint32_t *bf_pos0, uint64_t n_bf_lines, vgb_index_view *out)
{
	if (!c || !device_genome || !cstart || !clen || !out || n_contigs == 0) return VGB_E_ARG;
	if (n_snp_lines && (!snp_pos0 || !snp_code || !snp_rf || !snp_af)) return VGB_E_ARG;
	if (n_bf_lines && !bf_pos0) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return build_index_device(c, device_genome, genome_len, cstart, clen, n_contigs, snp_pos0, snp_code, snp_rf, snp_af, n_snp_lines,
	                          bf_pos0, n_bf_lines, out);
}

int vgb_build_ref_lite_bf_device(vgb_ctx *c, const uint8_t *device_genome, const uint64_t *cstart, const uint64_t *clen, uint32_t n_contigs,
                                 uint64_t **device_words, uint64_t *bits, uint64_t *nwords)
{
	if (!c || !device_genome || !cstart || !clen || !device_words || !bits || !nwords) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return build_ref_lite_bf(c, device_genome, cstart, clen, n_contigs, device_words, bits, nwords);
}

int vgb_build_snp_bf_ucsc_device(vgb_ctx *c, const uint8_t *device_genome, const uint32_t *pos0, const uint8_t *alt_code, uint64_t n_lines,
                                 uint64_t **device_words, uint64_t *bits, uint64_t *nwords)
{
	if (!c || !device_genome || !device_words || !bits || !nwords || (n_lines && (!pos0 || !alt_code))) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return build_snp_bf_ucsc(c, device_genome, pos0, alt_code, n_lines, device_words, bits, nwords);
}

void vgb_free_index_device(vgb_ctx *c, vgb_index_view *view)
{
	if (!c || !view) return;
	cudaSetDevice(c->device);
	free_index_device(view);
}

int vgb_index_upload_device(vgb_ctx *c, const vgb_index_view *device_view)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	c->upload_from_device = true;
	const int rc = index_upload(c, device_view);
	c->upload_from_device = false;
	return rc;
}

int vgb_synth_genome_device(vgb_ctx *c, uint8_t *device_out, const uint64_t *cstart, const uint64_t *clen, uint32_t n_contigs, uint64_t seed)
{
	if (!c || !device_out || !cstart || !clen) return VGB_E_ARG;
	cudaSetDevice(c->device);
	return synth_genome(c, device_out, cstart, clen, n_contigs, seed);
}

void *vgb_device_alloc(vgb_ctx *c, uint64_t bytes)
{
	if (!c) return nullptr;
	cudaSetDevice(c->device);
	void *p = nullptr;
	if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) { set_err(c, VGB_E_CUDA, "cudaMalloc(%llu) failed", (unsigned long long)bytes); return nullptr; }
	return p;
}

void vgb_device_free(vgb_ctx *c, void *p)
{
	if (!c) return;
	cudaSetDevice(c->device);
	cudaFree(p);
}

int vgb_memcpy_d2h(vgb_ctx *c, void *dst, const void *src, uint64_t bytes)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	VGB_CUDA(c, cudaStreamSynchronize(c->stream));
	VGB_CUDA(c, vgb::copy_sync(c, dst, src, bytes, cudaMemcpyDeviceToHost));
	return VGB_OK;
}

int vgb_memcpy_d2d(vgb_ctx *c, void *dst, const void *src, uint64_t bytes)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	VGB_CUDA(c, vgb::copy_sync(c, dst, src, bytes, cudaMemcpyDeviceToDevice));
	return VGB_OK;
}

int vgb_memset_device(vgb_ctx *c, void *dst, int value, uint64_t bytes)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	VGB_CUDA(c, vgb::memset_sync(c, dst, value, bytes));
	return VGB_OK;
}

int vgb_memcpy_h2d(vgb_ctx *c, void *dst, const void *src, uint64_t bytes)
{
	if (!c) return VGB_E_ARG;
	cudaSetDevice(c->device);
	VGB_CUDA(c, vgb::copy_sync(c, dst, src, bytes, cudaMemcpyHostToDevice));
	return VGB_OK;
}

}  // extern "C"
