// Host build of the VCF template and splice (vargeno_b200/csrc/vgb_vcf.cuh): test harness only, loaded by
// tests/test_vcf_template_host.py through ctypes and compared with `vargeno-b200 vcf-rewrite`.  Not part of libvgb200.so.
#include <cmath>
#include <cstdlib>

#include "../../vargeno_b200/csrc/vgb_vcf.cuh"

// contigs: names separated by '\n'; per site: 1-based concatenated position (ascending), gtype 0..3, confidence.  GQ is
// (int)(-1 * 10 * log(conf)) as the command line computes it.  Returns 0 and the VCF in *out (free with vgb_host_free), a
// VCF_E_* code with its message in err[0 .. 256), or -1 when the template cannot be built.
extern "C" int vgb_host_vcf_splice(const char *vcf, unsigned long long n, const char *names, const unsigned long long *lens, unsigned n_contigs,
                                   const unsigned *pos, const unsigned char *gt, const double *conf, unsigned long long n_sites, char **out,
                                   unsigned long long *out_len, char *err)
{
	std::vector<std::string> nm;
	std::vector<uint64_t> ln(lens, lens + n_contigs);
	for (const char *p = names; nm.size() < n_contigs; p++) {
		const char *e = strchr(p, '\n');
		nm.emplace_back(p, e ? (size_t)(e - p) : strlen(p));
		if (!e) break;
		p = e;
	}
	vgb::VcfTemplate t;
	std::string e;
	if (!vgb::vcf_template_parse(vcf, n, nm, ln, pos, n_sites, t, e)) { snprintf(err, 256, "%s", e.c_str()); return -1; }
	std::string text(vcf, n);
	text += t.extra;
	std::vector<int32_t> gq(n_sites);
	for (uint64_t i = 0; i < n_sites; i++) gq[i] = (int)(-1 * 10 * std::log(conf[i]));
	std::string o;
	const int rc = vgb::vcf_splice_host((const uint8_t *)text.data(), t, gt, gq.data(), o);
	if (rc) { snprintf(err, 256, "%s", vgb::vcf_error_text(rc)); return rc; }
	*out = (char *)malloc(o.size() + 1);
	memcpy(*out, o.data(), o.size());
	*out_len = o.size();
	return 0;
}

extern "C" void vgb_host_free(char *p) { free(p); }
