"""GPU parity: the CUDA path (through the C ABI of libvgb200.so) against the CPU oracle on the same inputs, and
against the golden outputs of the compiled reference (tests/golden).  Bit-exact for k-mer hits, votes, pileup
counts, genotypes; confidence must be bit-identical too (same host libm tables, same IEEE operation order), which
is stricter than the 1e-9 relative the spec asks for."""
import os

import numpy as np
import pytest

from oracle import oracle as orc

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
NAMES = ["s0", "advA", "advB"]


@pytest.fixture(scope="module")
def runs(cache):
    """name -> (Genotyper after the whole FASTQ, oracle after the whole FASTQ, oracle per-read results)."""
    from vargeno_b200.geno import Genotyper
    made = {}

    def get(name):
        if name not in made:
            ix = cache.index(name)
            fq = np.fromfile(cache.dataset(name).fastq, dtype=np.uint8)
            g = Genotyper(device=0, trace=True, max_chunk_bytes=1 << 20)    # small chunks: many submits, both slots
            g.upload_index(ix)
            g.submit(fq)
            g.sync()
            o = orc.Oracle(ix)
            res = o.process_fastq(fq)
            made[name] = (g, o, res)
        return made[name]
    yield get
    for g, o, _ in made.values():
        g.close()
        o.close()


@pytest.mark.parametrize("name", NAMES)
def test_static_sites_match(runs, name):
    g, o, _ = runs(name)
    s, os_ = g.sites(), o.sites()
    assert s["pos"].size == os_.size
    for a, b in (("pos", "pos"), ("ref", "ref"), ("alt", "alt"), ("ref_freq", "ref_freq"), ("alt_freq", "alt_freq")):
        assert np.array_equal(s[a], os_[b]), a


@pytest.mark.parametrize("name", NAMES)
def test_per_read_votes_match(runs, name):
    g, _, ores = runs(name)
    res = g.read_results()
    gold = np.load(os.path.join(GOLD, name + ".npz"))["reads"]
    assert res.size == ores.size == gold.size
    for f in ("flags", "freq", "n_ref", "n_snp", "passes", "ctx_hash"):
        bad = np.flatnonzero(res[f] != ores[f])
        assert bad.size == 0, "%s differs from the oracle for %d reads, first %s" % (f, bad.size, bad[:5])
    placed = (ores["flags"] & orc.F_PROCESS) != 0
    assert np.array_equal(res["target"][placed], ores["target"][placed])
    # and against the compiled reference's own trace
    for f in ("flags", "freq", "n_ref", "n_snp", "ctx_hash"):
        assert np.array_equal(res[f], gold[f]), f
    assert np.array_equal(res["target"][placed], gold["target"][placed])


@pytest.mark.parametrize("name", NAMES)
def test_pileup_counts_match(runs, name):
    g, o, _ = runs(name)
    r, a = g.pileup()
    os_ = o.sites()
    assert np.array_equal(r, os_["ref_cnt"]) and np.array_equal(a, os_["alt_cnt"])
    gold = np.load(os.path.join(GOLD, name + ".npz"))["sites"]
    assert np.array_equal(r, gold["ref_cnt"]) and np.array_equal(a, gold["alt_cnt"])


@pytest.mark.parametrize("name", NAMES)
def test_calls_match(runs, name):
    g, o, _ = runs(name)
    gt, conf = g.call()
    os_ = o.sites()
    exp_gt = np.zeros(os_.size, np.uint8)
    exp_cf = np.zeros(os_.size, np.float64)
    for i, s in enumerate(os_):
        if s["ref"] != s["alt"]:
            exp_gt[i], exp_cf[i] = orc.call(int(s["ref_cnt"]), int(s["alt_cnt"]), int(s["ref_freq"]), int(s["alt_freq"]))
    assert np.array_equal(gt, exp_gt)
    assert np.array_equal(conf, exp_cf), "confidence must be bit-identical (max rel err %g)" % np.max(
        np.abs(conf - exp_cf) / np.where(exp_cf == 0, 1, exp_cf))
    gold = np.load(os.path.join(GOLD, name + ".npz"))
    called = gt != 0
    assert np.array_equal(gt[called], gold["call_gt"]) and np.array_equal(conf[called], gold["call_conf"])


@pytest.mark.parametrize("name", NAMES)
def test_lookup_counters_match(runs, name):
    """The k-mer lookup metric is counted the same way on both sides (SURVEY.md 8(d))."""
    g, o, _ = runs(name)
    gs, os_ = g.stats(), o.stats()
    for k in ("reads", "skipped_n", "passes", "placed", "exact_lookups", "nbr_query_lookups", "nbr_scan_reads", "bf_probes",
              "lowq_kmers", "events", "pileup_incr", "big_kmers"):
        assert gs[k] == os_[k], (k, gs[k], os_[k])


@pytest.mark.parametrize("name", NAMES)
def test_probe_batch_matches(runs, cache, name):
    g, o, _ = runs(name)
    ix = cache.index(name)
    rng = np.random.default_rng(5)
    parts = [rng.integers(0, 1 << 63, 4000, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, 4000, dtype=np.uint64),
             ix.ref["kmer"][rng.integers(0, ix.ref.size, 4000)], ix.snp["kmer"][rng.integers(0, ix.snp.size, 2000)],
             np.array([0, 0xFFFFFFFFFFFFFFFF, 0xFFFFFFFF00000000, 0x00000000FFFFFFFF, ix.ref["kmer"][0], ix.ref["kmer"][-1],
                       ix.snp["kmer"][0], ix.snp["kmer"][-1]], dtype=np.uint64)]
    # one-base neighbours of dictionary k-mers
    base = ix.ref["kmer"][rng.integers(0, ix.ref.size, 2000)]
    sh = (rng.integers(0, 32, 2000) * 2).astype(np.uint64)
    parts.append(base ^ (rng.integers(1, 4, 2000).astype(np.uint64) << sh))
    kmers = np.concatenate(parts).astype(np.uint64)
    hits = g.lookup(kmers)
    for i, km in enumerate(kmers):
        km = int(km)
        r = o.lookup(0, km)
        s = o.lookup(1, km)
        rlo, rn, slo, sn = o.blocks(km)
        h = hits[i]
        assert bool(h["ref_found"]) == (r is not None) and bool(h["snp_found"]) == (s is not None), hex(km)
        if r is not None:
            assert (int(h["ref_pos"]), int(h["ref_flag"])) == (r[0], r[1]), hex(km)
        if s is not None:
            assert (int(h["snp_pos"]), int(h["snp_flag"]), int(h["snp_info"])) == s, hex(km)
        assert int(h["ref_block_n"]) == rn and int(h["snp_block_n"]) == sn
        if rn:
            assert int(h["ref_block_lo"]) == rlo
        if sn:
            assert int(h["snp_block_lo"]) == slo
        assert int(h["ref_bf"]) == o.bf_check(0, km & 0xFFFFFFFF) and int(h["snp_bf"]) == o.bf_check(1, km & 0xFFFFFFFFFF)


def test_resident_input_and_pinned_paths_agree(cache):
    """vgb_submit_fastq_device (input already in HBM) and the pinned double-buffer path give the same counters as
    the plain host-pointer path."""
    from vargeno_b200.geno import Genotyper
    ix = cache.index("s0")
    fq = np.fromfile(cache.dataset("s0").fastq, dtype=np.uint8)
    with Genotyper(device=0, max_chunk_bytes=8 << 20) as g:
        g.upload_index(ix)
        g.submit(fq)
        g.sync()
        ref = g.pileup()
        st = g.stats()
        # resident
        g.reset()
        d = g.dalloc(fq.size)
        g.h2d(d, fq)
        g.submit_device(d, fq.size)
        g.sync()
        got = g.pileup()
        assert np.array_equal(ref[0], got[0]) and np.array_equal(ref[1], got[1])
        assert g.stats()["exact_lookups"] == st["exact_lookups"]
        g.dfree(d)
        # pinned slots
        g.reset()
        chunks = Genotyper.split_records(fq, 2 << 20)
        for i, (s, e, n) in enumerate(chunks):
            buf = g.pinned_buffer(i & 1)
            buf[:e - s] = fq[s:e]
            g.submit_pinned(i & 1, e - s)
        g.sync()
        got = g.pileup()
        assert np.array_equal(ref[0], got[0]) and np.array_equal(ref[1], got[1])


def test_format_violations_are_loud(cache):
    from vargeno_b200.geno import Genotyper, VgbError
    ix = cache.index("s0")
    good = b"@r1\n" + b"ACGT" * 10 + b"\n+\n" + b"I" * 40 + b"\n"
    cases = {
        "truncated record": good + b"@r2\nACGT\n",
        "invalid base": b"@r1\n" + b"ACGU" * 10 + b"\n+\n" + b"I" * 40 + b"\n",
        "short quality": b"@r1\n" + b"ACGT" * 16 + b"\n+\n" + b"I" + b"\n",
    }
    for what, text in cases.items():
        with Genotyper(device=0) as g:
            g.upload_index(ix)
            g.submit(text)
            with pytest.raises(VgbError) as ei:
                g.sync()
            assert ei.value.code == -3, what
    with Genotyper(device=0) as g:      # N is not an error: the read is skipped (src/qv.cc:815-828)
        g.upload_index(ix)
        g.submit(b"@r1\n" + b"ACGN" * 10 + b"\n+\n" + b"I" * 40 + b"\n" + good)
        g.sync()
        st = g.stats()
        assert st["reads"] == 2 and st["skipped_n"] == 1


def test_long_reads_and_context_overflow_take_the_deferred_path(cache):
    """Reads of 288+ bases (more than 8 k-mers) and reads with more hit contexts than the group kernels (4 or 8 lanes per read) keep in shared
    memory are handed on: up to 64 contexts per pass to the wide-list instantiation (8 lanes per read), beyond that and beyond 8 k-mers to the
    last stage (32 lanes, one read per warp, contexts spilled to global memory); results must not depend on which kernel handled a read."""
    from vargeno_b200.geno import Genotyper
    from vargeno_b200.tools import synth
    import datasets
    ix = cache.index("advB")
    # rebuild the advB genome/haplotypes (pure function of its seeds) and draw long reads from it
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        ds = datasets.make_adv_b(d)
        names, seqs = [], []
        from vargeno_b200.tools import index_builder as ib
        names, seqs = ib.read_fasta_raw(ds.fasta)
    g0 = synth.Genome(names, seqs)
    haps = (g0.concat(), g0.concat())
    parts, first = [], 0
    for L, n in ((288, 600), (320, 600), (650, 400), (1000, 300), (150, 800), (100, 400)):
        parts.append(synth.simulate_reads(g0, haps, n, L, seed=77 + L, sub_rate=0.01, lowq_prob=0.7, lowq_chars=31, first_id=first))
        first += n
    # reverse-strand 150 bp reads over the 6-copy repeat family, all leading qualities low: the forward pass finds nothing, the
    # retry finds 6 positions per k-mer (24 exact contexts) plus neighbours -> more than the group kernels keep
    gb = datasets.adv_b_genome()
    rs = np.array([o + d for (_, _, ci, o, l) in gb.repeat_copies if l == 250 for d in (0, 7, 33, 64, 100)] * 4, dtype=np.int64)
    assert rs.size >= 100
    n_before_retry_set = first
    parts.append(synth.simulate_reads(gb, (gb.concat(), gb.concat()), rs.size, 150, seed=91, sub_rate=0.002, lowq_prob=1.0, lowq_chars=4,
                                      first_id=first, forced_starts=rs, forced_rev=np.ones(rs.size, bool)))
    first += rs.size
    fq = np.concatenate(parts)
    o = orc.Oracle(ix)
    want = o.process_fastq(fq)
    with Genotyper(device=0, trace=True, max_chunk_bytes=1 << 20) as g:
        g.upload_index(ix)
        g.submit(fq)
        g.sync()
        got = g.read_results()
        r, a = g.pileup()
        st = g.stats()
    for f in ("flags", "freq", "n_ref", "n_snp", "passes", "ctx_hash"):
        bad = np.flatnonzero(got[f] != want[f])
        assert bad.size == 0, "%s differs for %d reads, first %s" % (f, bad.size, bad[:5])
    sites = o.sites()
    assert np.array_equal(r, sites["ref_cnt"]) and np.array_equal(a, sites["alt_cnt"])
    ost = o.stats()
    for k in ("reads", "passes", "placed", "exact_lookups", "nbr_query_lookups", "nbr_scan_reads", "events", "pileup_incr", "big_kmers"):
        assert st[k] == ost[k], k
    n_ctx = want["n_ref"].astype(int) + want["n_snp"].astype(int)
    assert int(np.count_nonzero((n_ctx > 24) & (n_ctx <= 64))) > 0, "the set should contain reads for the wide-list kernel (25..64 contexts in a pass)"
    assert int(n_ctx.max()) > 64, "the set should contain reads beyond the wide list as well (last stage, spilled contexts)"
    # short reads (<= 8 k-mers) whose RETRY pass overflows the budget: the 4-lane kernel has already run and accounted for their
    # forward pass and hands over only the retry (bit 31 of the deferred-list entry)
    short = np.arange(want.size) >= n_before_retry_set
    n_retry_overflow = int(np.count_nonzero(short & (want["passes"] == 2) & (want["n_ref"].astype(int) + want["n_snp"].astype(int) > 24)))
    assert n_retry_overflow > 0, "the set should contain short reads that overflow in the retry pass"
    o.close()
    # the chain without the wide-list kernel gives the same answer: the 25..64-context reads then go to the last stage as well
    os.environ["VGB_NO_WIDE"] = "1"
    try:
        with Genotyper(device=0, trace=True, max_chunk_bytes=1 << 20) as g:
            g.upload_index(ix)
            g.submit(fq)
            g.sync()
            got2 = g.read_results()
            st2 = g.stats()
    finally:
        os.environ.pop("VGB_NO_WIDE", None)
    assert np.array_equal(got, got2)
    for k in ("reads", "passes", "placed", "exact_lookups", "nbr_query_lookups", "nbr_scan_reads", "events", "pileup_incr", "big_kmers"):
        assert st2[k] == st[k], k


def test_device_read_simulator_matches_numpy(cache):
    """vgb_synth_reads_device is the bench's input generator; it must emit the bytes tools/synth.simulate_reads does."""
    from vargeno_b200.geno import Genotyper
    from vargeno_b200.tools import synth
    g0 = synth.make_genome([("chrA", 50000), ("chrB", 30000)], seed=3, n_runs=[(0, 1000, 50)])
    snps = synth.make_snps(g0, 100, seed=3)
    h0, h1 = synth.donor_haplotypes(g0, snps, seed=3)
    want = synth.simulate_reads(g0, (h0, h1), 3000, 150, seed=9, sub_rate=0.01, lowq_prob=0.3, first_id=12345)
    with Genotyper(device=0) as g:
        d0, d1, out = g.dalloc(h0.size), g.dalloc(h1.size), g.dalloc(want.size)
        g.h2d(d0, h0)
        g.h2d(d1, h1)
        g.synth_reads_device(d0, d1, h0.size, g0.starts, g0.lengths, 3000, 150, 9, 12345, 9, 0.01, 0.3, 4, out, want.size)
        got = g.d2h(out, want.size)
    assert np.array_equal(got, want)
