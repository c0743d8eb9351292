#!/usr/bin/env python
"""bench.py -- reads/s (and k-mer lookups/s) of the `vargeno geno` hot path on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W]              our CUDA path (one rank per GPU under torchrun)
    python bench.py --impl reference [--steps K] [--warmup W]        the reference's own CPU geno on the host cores

Default workload = the configuration BASELINE.json's metric is quoted on ("synthetic 150bp WGS reads"): configs[2],
SURVEY.md 8(d) "S2": GRCh38-shaped 3.1 Gbp reference (24 contigs, 5 % N, 2 % planted repeats), 12 M-SNP list, 150 bp reads at
0.5 % substitutions, first four quality characters below '8' with probability 0.25.  It fits one GPU (~106 GB of HBM).
`--workload s1` = configs[1] (chr22-shaped), `--workload s3` = configs[3] (2 % substitutions, all leading qualities low).
With the default workload the same JSON line also carries, under "shapes", the S3 stress reads and the S4 dictionary-probe
microbenchmark (configs[4], 38 launches of 2^28 k-mers = 10^10 per probe set) against the same index, at every N.

One step = one batch of `--batch-reads` FASTQ records (default 2 M = 632 MB of text) through the whole per-read path
(framing, 2-bit packing, exact + Hamming-1 lookups, Bloom gates, vote, pileup atomics).  Every step gets a distinct
batch that is larger than the 126 MB L2, so no L2 flush is needed between steps.

Timed regions are bracketed by a barrier and a device synchronise on both sides (max over ranks); the kernel time for the
roofline comes from CUDA events recorded on the launching stream inside libvgb200.so.  A multi-rank run checks its own
result: rank 0 re-processes every rank's batches on its own GPU and compares the raw counters and the calls with what the
NCCL all-reduce left ("parity_checked"); a mismatch exits non-zero.

`--dump-outputs DIR` writes what the HBM-resident leg (the one `value` is quoted on) left behind after its last step -- per-site
counters and calls, on a seeded sample of the sites when there are more than DUMP_SITES, and the counters of the timed steps --
as float32 / float64 .npy files.  Index and reads are generated from fixed seeds, so two builds run with the same arguments on
the same workload (the line's config.workload) can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

REC_ID_WIDTH = 9
LOWQ_CHARS = 4
READ_LEN = 150
# sub_rate, lowq_prob of the read sets (SURVEY.md 8(d))
READ_SETS = {"s1": (0.005, 0.25), "s2": (0.005, 0.25), "s3": (0.02, 1.0)}
# the reference arm leaves this behind when it could not run the GRCh38-shaped workload (memory / start-up time): our arm then
# runs S1 as well, so that the two arms of one driver run are never on different workloads
FALLBACK_MARK = "/tmp/vgb200_bench_workload_fallback"
KERNEL_SOURCES = ["vargeno_b200/csrc/vgb_geno8.inl", "vargeno_b200/csrc/vgb_geno.cu", "vargeno_b200/csrc/vgb_common.cuh",
                  "vargeno_b200/csrc/vgb_index.cu"]
# --dump-outputs: at most this many SNP sites are written (a fixed, seeded sample of the GRCh38-shaped list keeps the files near
# 28 MB); the counters are the ones tests compare with the oracle (timings and chunk bookkeeping left out)
DUMP_SITES = 1 << 20
DUMP_COUNTERS = ("reads", "skipped_n", "passes", "placed", "exact_lookups", "nbr_query_lookups", "nbr_scan_reads", "bf_probes",
                 "lowq_kmers", "events", "pileup_incr", "big_kmers")


def rec_bytes(read_len=READ_LEN):
    return 2 + REC_ID_WIDTH + 1 + read_len + 3 + read_len + 1


def kernel_hash():
    h = hashlib.sha256()
    for f in KERNEL_SOURCES:
        h.update(open(os.path.join(ROOT, f), "rb").read())
    return h.hexdigest()[:16]


def ncu_constants(workload):
    """Per-launch counters of the dominant kernel from a committed `ncu --set full` capture (profiles/ncu_constants.json):
    a number taken under the profiler cannot be measured in the timed run, so it is a constant -- tied to a hash of the
    kernel sources, so that it reads `stale` (and the keys derived from it read null) after the next kernel change instead of
    silently describing an older build."""
    p = os.path.join(ROOT, "profiles", "ncu_constants.json")
    try:
        all_c = json.load(open(p))
    except Exception:
        return None
    c = all_c.get(workload)
    if not c:
        return None
    c = dict(c)
    c["stale"] = c.get("kernel_hash") != kernel_hash()
    return c


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def mem_available_gb():
    try:
        return int([l for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0].split()[1]) / 1e6
    except Exception:
        return 0.0


def workload_config(workload, scale, name, counts, n_sites):
    """The `config` object: what defines the workload and nothing else, so that both arms print the same one."""
    sub, lowq = READ_SETS[workload]
    return {"workload": "%s, %s, %dbp reads @%g%% subst, lowq %g on first %d quality chars" % (
                name, "1M-SNP list" if workload == "s1" else "12M-SNP list", READ_LEN, sub * 100, lowq, LOWQ_CHARS),
            "baseline_config": {"s1": "configs[1]", "s2": "configs[2]", "s3": "configs[3]"}[workload], "scale": scale,
            "read_len": READ_LEN, "ref_kmers": counts["ref_kmers"], "snp_kmers": counts["snp_kmers"], "snp_sites": int(n_sites),
            "index": "replicated per GPU, built by vgb_build_index_device (byte-identical to `vargeno index`)",
            "reads": "sharded across GPUs", "l2": "every step streams a distinct batch larger than L2 (no flush needed)"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""

    def __init__(self, device):
        super().__init__(daemon=True)
        self.device = device
        self.rows = []
        self.stop_flag = threading.Event()
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag.is_set():
                    break
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag.set()
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def bind_near_gpu(device):
    """Run this rank on the CPUs NVML names as closest to its GPU, so that the pinned FASTQ buffers (first touched by this
    process) sit in host memory of the same NUMA node as the GPU's PCIe root.  Returns what was done, for the JSON line."""
    nodes = "?"
    try:
        nodes = open("/sys/devices/system/node/online").read().strip()
    except Exception:
        pass
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1]
        cpus = [c for c in cpus if c < ncpu]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return ("cpus %d-%d" % (min(cpus), max(cpus)) if len(cpus) > 1 else "cpu %d" % cpus[0]) + ", numa nodes online: " + nodes
    except Exception as e:     # best effort: the number is still valid without it, only possibly slower
        return "unbound (%s), numa nodes online: %s" % (type(e).__name__, nodes)
    return "unbound, numa nodes online: " + nodes


def build_workload(g, workload, scale, keep_host=False):
    from vargeno_b200.tools import device_workloads as dw
    if workload == "s1":
        return dw.build_s1(g, scale=scale, keep_host=keep_host)
    # BASELINE.json configs[2] / [3] (SURVEY.md 8(d) S2 / S3): GRCh38-shaped reference, 12 M SNPs; same index for both
    contigs = [(n, max(64, int(l * scale))) for n, l in dw.GRCH38]
    return dw.build(g, contigs, max(100, int(12_000_000 * scale)), seed=38, name="S2 GRCh38-shaped x%g" % scale, keep_host=keep_host)


def lookups(st):
    return st["exact_lookups"] + st["nbr_query_lookups"] + st["nbr_scan_reads"]


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from vargeno_b200.geno import Genotyper
    from vargeno_b200.tools import device_workloads as dw

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_near_gpu(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    workload, fallback_note = args.workload, None
    if workload != "s1" and os.path.exists(FALLBACK_MARK):
        fallback_note = "reference arm fell back to S1 on this box (%s): this arm follows" % open(FALLBACK_MARK).read().strip()
        workload = "s1"
    K, W, B = args.steps, args.warmup, args.batch_reads
    t_setup = time.time()
    L = READ_LEN
    rb = rec_bytes(L)
    batch_bytes = B * rb
    nb = K + W

    uid = None
    if world > 1:
        box = [Genotyper.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        uid = box[0]
    g = Genotyper(device=local, max_chunk_bytes=batch_bytes + 4096, world_size=world, rank=rank, nccl_unique_id=uid)
    # index: genome text, SNP list, reference-format index records and the GPU re-layout, all produced through the device
    # (vgb_build_index_device is byte-identical to `vargeno index`: tests/test_gpu_index_build.py); replicated on every rank
    want_cpu = rank == 0 and world == 1 and not args.skip_cpu
    cpu_skip = None
    if want_cpu and workload != "s1" and args.scale >= 0.5 and mem_available_gb() < 150:
        want_cpu, cpu_skip = False, "oracle port skipped: %.0f GB of host memory available, the GRCh38-sized index image + the oracle's arrays need ~130 GB" % mem_available_gb()
    wl = build_workload(g, workload, args.scale, keep_host=want_cpu)
    if world > 1:
        g.allreduce()                       # NCCL connection set-up happens on the first collective: keep it out of the timed legs

    # synthetic reads, generated on the device (byte-identical twin of tools/synth.simulate_reads)
    d_reads = g.dalloc(nb * batch_bytes)
    first = rank * nb * B
    sub_rate, lowq_prob = READ_SETS[workload]
    dw.synth_batch(g, wl, d_reads, nb * B, first, sub_rate, lowq_prob, LOWQ_CHARS, REC_ID_WIDTH)
    # host copy in pinned memory for the end-to-end leg
    pinned = torch.empty(nb * batch_bytes, dtype=torch.uint8, pin_memory=True)
    host = pinned.numpy()
    for i in range(nb):                     # batch by batch: no second copy of the whole read set in host memory
        host[i * batch_bytes:(i + 1) * batch_bytes] = g.d2h(d_reads + i * batch_bytes, batch_bytes)
    # pinned destination of the job's result (GT + confidence per SNP site), allocated once like a real caller would
    out_gt = torch.empty(g.n_sites, dtype=torch.uint8, pin_memory=True).numpy()
    out_conf = torch.empty(g.n_sites, dtype=torch.float64, pin_memory=True).numpy()
    setup_s = time.time() - t_setup

    def barrier():
        g.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def raw_counters():
        p, n = g.counter_device_ptr()
        return g.d2h(p, n * 4).view(np.uint32).copy()

    def resident_leg(d_buf, first_id):
        """W untimed + K timed steps over batches already in HBM; returns (seconds, stats before, stats after)."""
        g.reset()
        for i in range(W):
            g.submit_device(d_buf + i * batch_bytes, batch_bytes, first_id + i * B)
        barrier()
        s0 = g.stats()
        t0 = time.perf_counter()
        for i in range(W, nb):
            g.submit_device(d_buf + i * batch_bytes, batch_bytes, first_id + i * B)
        g.sync()
        if world > 1:
            g.allreduce()                   # the one exchange step of the job (NCCL sum of the per-SNP counters)
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        return dt, s0, g.stats()

    def e2e_leg(host_buf, first_id):
        """The same K steps through vgb_submit_fastq with HOST buffers: H2D inside the timed region, calls read back."""
        g.reset()
        for i in range(W):
            g.submit_chunk(host_buf[i * batch_bytes:(i + 1) * batch_bytes], first_id + i * B)
        g.sync()
        g.call(out=(out_gt, out_conf))      # warm-up of the result path too (its device staging is allocated at first use)
        barrier()
        t0 = time.perf_counter()
        for i in range(W, nb):
            g.submit_chunk(host_buf[i * batch_bytes:(i + 1) * batch_bytes], first_id + i * B)
        g.sync()
        t_reads = time.perf_counter() - t0
        if world > 1:
            g.allreduce()
        t_reduce = time.perf_counter() - t0 - t_reads
        g.call(out=(out_gt, out_conf))      # device -> host read of the job's result (GT + confidence per SNP site)
        t_call = time.perf_counter() - t0 - t_reads - t_reduce
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        return dt, {"submit_and_sync": t_reads * 1e3, "allreduce": t_reduce * 1e3, "call_d2h": t_call * 1e3}

    def leg_numbers(dt, s0, s1):
        reads = s1["reads"] - s0["reads"]
        d_look = lookups(s1) - lookups(s0)
        ms_geno = s1["gpu_ms_geno"] - s0["gpu_ms_geno"]
        ms_parse = s1["gpu_ms_parse"] - s0["gpu_ms_parse"]
        return {"value": K * B * world / dt, "ms_per_step": dt / K * 1e3, "lookups": d_look, "reads": reads, "ms_geno": ms_geno, "ms_parse": ms_parse,
                "lookups_per_read": d_look / max(1, reads), "placed_fraction": (s1["placed"] - s0["placed"]) / max(1, reads),
                "launches": s1["kernel_launches"] - s0["kernel_launches"],
                "kmer_lookups_per_s": sum_over_ranks(d_look) / dt}

    # ---- leg 1: inputs resident in HBM ----
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.5)                         # nvidia-smi needs a moment to come up; samples cover both timed legs
    dt, st0, st1 = resident_leg(d_reads, first)
    main = leg_numbers(dt, st0, st1)
    dump = job_outputs(g, st0, st1) if args.dump_outputs and rank == 0 else None

    # ---- kernel durations for the roofline: the same steps with every kernel alone on the GPU ----
    # In production the hand-over kernels of a chunk (a few thousand reads from repeat families, a long dependent chain each) run
    # on a second stream under the framing and the main kernel of the next chunk; their event intervals then overlap and cannot
    # be added up.  VGB_NO_TAIL_OVERLAP serialises them behind the main kernel (re-read by the library at vgb_reset_counts under
    # VGB_RETUNE): `value` above is the production mode, the roofline's launch_ms comes from this leg.
    os.environ["VGB_RETUNE"] = "1"
    os.environ["VGB_NO_TAIL_OVERLAP"] = "1"
    dts, ss0, ss1 = resident_leg(d_reads, first)
    serial = leg_numbers(dts, ss0, ss1)
    os.environ.pop("VGB_NO_TAIL_OVERLAP")       # every later leg starts with vgb_reset_counts, which puts the production mode back

    # ---- self-check of the multi-rank result (rank 0 redoes every rank's batches on its own GPU) ----
    parity = None
    if world > 1:
        reduced = raw_counters()            # after vgb_allreduce_pileup: the sum over ranks of all nb batches
        gt_red, conf_red = g.call()
        gt_red, conf_red = gt_red.copy(), conf_red.copy()
        ok = True
        if rank == 0:
            g.reset()
            for r in range(world):
                fr = r * nb * B
                dw.synth_batch(g, wl, d_reads, nb * B, fr, sub_rate, lowq_prob, LOWQ_CHARS, REC_ID_WIDTH)
                for i in range(nb):
                    g.submit_device(d_reads + i * batch_bytes, batch_bytes, fr + i * B)
                g.sync()
            alone = raw_counters()
            gt_one, conf_one = g.call()
            ok = bool(np.array_equal(alone, reduced) and np.array_equal(gt_one, gt_red) and np.array_equal(conf_one, conf_red))
            parity = {"parity_checked": ok, "n_sites_compared": int(g.n_sites), "reads_compared": int(world * nb * B),
                      "counter_sum": int(reduced.astype(np.uint64).sum()),
                      "how": "rank 0 re-processed all %d ranks' batches on one GPU: raw counters == NCCL all-reduced counters, vgb_call output identical" % world}
            dw.synth_batch(g, wl, d_reads, nb * B, first, sub_rate, lowq_prob, LOWQ_CHARS, REC_ID_WIDTH)   # own reads back in place
        flag = torch.tensor([1.0 if ok else 0.0], device="cuda")
        dist.broadcast(flag, src=0)
        if flag.item() != 1.0:
            if rank == 0:
                sys.stderr.write("bench.py: MULTI-RANK PARITY FAILURE: all-reduced counters differ from the single-GPU result\n")
                emit(dict(parity, metric="reads/s", value=None, n_gpus=world))
            sys.exit(3)

    # ---- leg 2: end to end through the C ABI with host buffers (H2D inside the timed region, calls read back) ----
    dt_e2e, e2e_ms = e2e_leg(host, first)
    e2e_value = K * B * world / dt_e2e

    # ---- what the host -> device path of this box delivers with nothing else going on (all ranks at once, no kernels) ----
    dst = torch.empty(batch_bytes, dtype=torch.uint8, device="cuda")
    for i in range(2):
        dst.copy_(pinned[i * batch_bytes:(i + 1) * batch_bytes], non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for i in range(W, nb):
        dst.copy_(pinned[i * batch_bytes:(i + 1) * batch_bytes], non_blocking=True)
    torch.cuda.synchronize()
    barrier()
    dt_copy = max_over_ranks(time.perf_counter() - t0)
    h2d_ceiling = K * batch_bytes * world / dt_copy / 1e9
    del dst

    # keep the GPU busy a little longer so that the 100 ms clock sampler sees the part under this load
    t_end = time.perf_counter() + args.clock_hold_s
    while time.perf_counter() < t_end:
        for i in range(nb):
            g.submit_device(d_reads + i * batch_bytes, batch_bytes, first + i * B)
        g.sync()
    clocks = sampler.finish()

    # ---- the other named shapes against the same index: S3 stress reads, S4 probe microbenchmark ----
    shapes = None
    rs = None
    if world == 1 and not args.skip_roofline_probe:
        try:
            rs = g.random_sector_bench(32 << 30, 1 << 30, 3)
        except Exception:
            rs = None
    if workload == "s2" and not args.skip_shapes:
        shapes = {}
        s3_sub, s3_lowq = READ_SETS["s3"]
        dw.synth_batch(g, wl, d_reads, nb * B, first, s3_sub, s3_lowq, LOWQ_CHARS, REC_ID_WIDTH)
        dt3, a0, a1 = resident_leg(d_reads, first)
        s3 = leg_numbers(dt3, a0, a1)
        for i in range(nb):
            host[i * batch_bytes:(i + 1) * batch_bytes] = g.d2h(d_reads + i * batch_bytes, batch_bytes)
        dt3e, _ = e2e_leg(host, first)
        shapes["s3"] = {"workload": workload_config("s3", args.scale, wl.name, wl.index_counts, g.n_sites)["workload"],
                        "value": s3["value"], "unit": "reads/s", "ms_per_step": s3["ms_per_step"], "e2e_value": K * B * world / dt3e,
                        "kmer_lookups_per_s": s3["kmer_lookups_per_s"], "lookups_per_read": s3["lookups_per_read"],
                        "placed_fraction": s3["placed_fraction"], "k_geno_ms_per_step": s3["ms_geno"] / K,
                        "algorithmic_gbs_rank0": s3["lookups"] * 32.0 / (s3["ms_geno"] * 1e-3) / 1e9 if s3["ms_geno"] > 0 else None}
        n_probe = max(1 << 16, int((1 << 28) * min(1.0, args.scale)))
        s4 = {}
        for mode, name in ((0, "uniform_random_misses"), (1, "sampled_dictionary_hits"), (2, "half_half")):
            barrier()
            ms, found = g.probe_bench(n_probe, mode, 11 + rank, args.probe_launches)
            ms = max_over_ranks(ms)
            lps = 2.0 * n_probe * world / (ms * 1e-3)
            s4[name] = {"kmers_per_launch_per_gpu": n_probe, "launches": args.probe_launches, "kmers_total": n_probe * args.probe_launches * world,
                        "ms_per_launch": ms, "lookups_per_s": lps, "found_per_launch_rank0": int(found),
                        "frac_of_random_sector_rate": (lps / world * 32.0 / 1e9 / rs) if rs else None}
        shapes["s4"] = {"workload": "dictionary-probe microbenchmark (BASELINE configs[4]): one reference + one SNP dictionary lookup per 32-mer against the same index",
                        "random_sector_peak_gbs": rs, "probe_sets": s4}

    out = None
    if rank == 0:
        cpu = None
        if want_cpu:
            sample = host_sample(g, wl, d_reads, min(B, args.cpu_sample), first, sub_rate, lowq_prob)
            stress_sample = None
            if workload == "s2" and not args.skip_shapes:          # the stress shape (every gate open, 2 % substitutions) on the same index
                stress_sample = host_sample(g, wl, d_reads, min(B, max(1, args.cpu_sample // 4)), first, READ_SETS["s3"][0], READ_SETS["s3"][1])
            cpu, st_o, sites_o, stress_o = cpu_port_baseline(wl.host_index, sample, stress_sample)
            cpu["parity"] = parity_against_port(g, sample, st_o, sites_o)
            if stress_o is not None:
                cpu["parity_s3"] = parity_against_port(g, stress_sample, stress_o[0], stress_o[1])
                cpu["parity"]["parity_checked"] = cpu["parity"]["parity_checked"] and cpu["parity_s3"]["parity_checked"]
            if not cpu["parity"]["parity_checked"]:
                sys.stderr.write("bench.py: PARITY FAILURE against the CPU port on the full-size index: %s\n" % json.dumps(cpu["parity"]))
                emit({"metric": "reads/s", "value": None, "n_gpus": world, "cpu_baseline": cpu})
                sys.exit(3)
        elif cpu_skip:
            cpu = {"value": None, "unit": "reads/s", "cores": 0, "kind": "port", "sample": cpu_skip}
        peak, peak_src = measured_peaks()
        alg_bytes = serial["lookups"] * 32.0
        achieved = alg_bytes / (serial["ms_geno"] * 1e-3) / 1e9 if serial["ms_geno"] > 0 else 0.0
        nc = ncu_constants(workload) if args.scale == 1.0 else None
        fresh = bool(nc) and not nc["stale"]
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": nc["dram_bytes_per_read"] * B if fresh else None,
                "kernel": "k_geno8 (+ the hand-over kernels behind it: wide-list stage, warp-per-read kernel)", "algorithmic_bytes_per_launch": alg_bytes / K,
                "launch_ms": serial["ms_geno"] / K,
                "launch_ms_note": "CUDA events on the kernel stream with the hand-over kernels serialised behind the main kernel (VGB_NO_TAIL_OVERLAP); "
                                  "`value` runs them on a second stream under the next chunk's kernels",
                "serial_reads_per_s": serial["value"],
                "peak_source": peak_src, "note": "achieved = 32 B (one DRAM sector) per dictionary lookup (SURVEY.md 8(d)) / CUDA-event kernel time; "
                "the physical figures are the request-rate keys below",
                "random_sector_peak_gbs": rs, "random_loads_per_s_peak": rs * 1e9 / 32 if rs else None}
        if nc:
            roof["ncu"] = {k: nc.get(k) for k in ("source", "kernel_hash", "stale", "reads_per_launch")}
        if fresh:
            reads_per_s_kernel = B / (serial["ms_geno"] / K * 1e-3)
            roof["l2_requests_per_read"] = nc["l2_requests_per_read"]
            roof["dram_fetches_per_read"] = nc["dram_fetches_per_read"]
            if rs:
                # one random load of the denominator probe = one L2 request = one DRAM fetch: the physical fractions
                roof["request_rate_frac"] = nc["l2_requests_per_read"] * reads_per_s_kernel / (rs * 1e9 / 32)
                roof["dram_fetch_rate_frac"] = nc["dram_fetches_per_read"] * reads_per_s_kernel / (rs * 1e9 / 32)
        out = {
            "metric": "reads/s", "value": main["value"], "unit": "reads/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": workload_config(workload, args.scale, wl.name, wl.index_counts, g.n_sites),
            "batch": {"reads_per_step_per_gpu": B, "fastq_bytes_per_step_per_gpu": batch_bytes},
            "kmer_lookups_per_s": main["kmer_lookups_per_s"],
            "lookups_per_read": main["lookups_per_read"],
            "placed_fraction": main["placed_fraction"],
            "roofline": roof,
            "kernel_ms_per_step": {"k_geno": serial["ms_geno"] / K, "fastq_framing": serial["ms_parse"] / K,
                                   "overlapped_event_sums": {"k_geno": main["ms_geno"] / K, "fastq_framing": main["ms_parse"] / K}},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": batch_bytes * world,
                    "d2h_bytes_per_step": int(g.n_sites * 9 * world / K), "ms_per_step": dt_e2e / K * 1e3, "rank0_ms": e2e_ms,
                    "h2d_achieved_gbs": K * batch_bytes * world / dt_e2e / 1e9,
                    "h2d_ceiling_gbs": h2d_ceiling,
                    "h2d_ceiling_note": "all ranks copying the same pinned batches at once, no kernels: what this box's host-to-device path delivers"},
            "gpu_launches": int(main["launches"]),
            "clocks": clocks,
            "host_binding": numa,
            "setup_s": setup_s,
        }
        if parity:
            out.update(parity)
        if shapes:
            out["shapes"] = shapes
        if fallback_note:
            out["workload_fallback"] = fallback_note
        if dump:
            out["dump_outputs"] = write_outputs(args.dump_outputs, dump)
        emit(out)
    g.dfree(d_reads)
    g.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


def host_sample(g, wl, d_buf, n, first_id, sub_rate, lowq_prob):
    """The first n reads of this rank's read set (the device buffer may hold another set by now: regenerate)."""
    from vargeno_b200.tools import device_workloads as dw
    dw.synth_batch(g, wl, d_buf, n, first_id, sub_rate, lowq_prob, LOWQ_CHARS, REC_ID_WIDTH)
    return g.d2h(d_buf, n * rec_bytes())


def job_outputs(g, s0, s1):
    """What a caller of the timed path holds after its last step: per-site ref / alt counters (all-reduced when N > 1) and the
    calls (GT code, confidence), on all sites or on a sorted sample of DUMP_SITES drawn with a fixed seed (the sample depends
    only on the site count, so two builds dump the same sites), plus the counters of the K timed steps."""
    ref_cnt, alt_cnt = g.pileup()
    gt, conf = g.call()
    n = ref_cnt.size
    idx = np.arange(n) if n <= DUMP_SITES else np.sort(np.random.default_rng(0).choice(n, DUMP_SITES, replace=False))
    return {"site_index": idx.astype(np.float64), "ref_cnt": ref_cnt[idx].astype(np.float32), "alt_cnt": alt_cnt[idx].astype(np.float32),
            "gt": gt[idx].astype(np.float32), "conf": conf[idx].astype(np.float64),
            "counters": np.array([s1[k] - s0[k] for k in DUMP_COUNTERS], dtype=np.float64)}


def write_outputs(d, arrays):
    """<d>/<name>.npy per array; returns what the JSON line says about it."""
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a)
    return {"dir": d, "files": sorted(name + ".npy" for name in arrays), "sites": int(arrays["site_index"].size),
            "bytes": int(sum(a.nbytes for a in arrays.values())), "counters": list(DUMP_COUNTERS)}


def cpu_port_baseline(index, text, stress_text=None):
    """Bounded single-thread run of the CPU oracle (kind "port") over a prefix of the same reads.  stress_text: a (smaller) sample
    of the stress read set, run untimed afterwards on the same oracle instance for the parity check of that shape."""
    from oracle import oracle as orc
    t0 = time.perf_counter()
    o = orc.Oracle(index)
    t_load = time.perf_counter() - t0
    t0 = time.perf_counter()
    o.process_fastq(np.ascontiguousarray(text), want_results=False)
    dt = time.perf_counter() - t0
    st = o.stats()
    sites = o.sites()
    stress = None
    if stress_text is not None:
        o.reset()
        o.process_fastq(np.ascontiguousarray(stress_text), want_results=False)
        stress = (o.stats(), o.sites())
    o.close()
    return {"value": st["reads"] / dt, "unit": "reads/s", "cores": 1, "kind": "port",
            "sample": "first %d reads of step 0, oracle/liboracle.so single thread, index resident (image copied back from the GPU once, "
                      "oracle arrays built in %.0f s, outside the timed %.1f s)" % (st["reads"], t_load, dt),
            "kmer_lookups_per_s": (st["exact_lookups"] + st["nbr_query_lookups"] + st["nbr_scan_reads"]) / dt}, st, sites, stress


def parity_against_port(g, text, st_o, sites_o):
    """The sample the CPU port just processed, through the CUDA path on the full-size index: every per-site counter (saturated
    like the reference's, src/vartype.h:27) and every lookup / placement counter must be the port's.  The checker's verdict goes
    into the line; a mismatch ends the run."""
    g.reset()
    g.submit_chunk(np.ascontiguousarray(text))         # one call: the sample is smaller than a batch
    g.sync()
    r, a = g.pileup()
    st = g.stats()
    keys = ("reads", "passes", "placed", "skipped_n", "exact_lookups", "nbr_query_lookups", "nbr_scan_reads", "events", "pileup_incr", "big_kmers")
    bad = [k for k in keys if k in st_o and int(st[k]) != int(st_o[k])]
    same = bool(np.array_equal(r, sites_o["ref_cnt"]) and np.array_equal(a, sites_o["alt_cnt"]))
    return {"parity_checked": same and not bad, "sites_compared": int(sites_o.size), "sites_with_counts": int(np.count_nonzero(r | a)),
            "reads_compared": int(st["reads"]), "counters_differing": bad,
            "how": "the CPU port's sample through the CUDA path on the same full-size index: per-site ref/alt counters and the read / pass / "
                   "placement / lookup / context / increment counters compared"}


# ------------------------------------------------------------------------------------------------------------------
# reference arm: the unmodified reference binary, one process per host core that fits in RAM, fed through FIFOs
# ------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import shutil
    import tempfile

    from oracle import oracle as orc
    from vargeno_b200.tools import index_builder as ib
    from vargeno_b200.tools import synth, workloads

    K, W = args.steps, args.warmup
    L = READ_LEN
    Bp = args.ref_batch_reads
    nb = K + W
    bb = Bp * rec_bytes(L)
    workload = args.workload
    try:
        os.remove(FALLBACK_MARK)
    except OSError:
        pass
    fallback = None
    have_gpu = False
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        pass
    # per-process memory of the reference: 9 B x ref entries + 16 GiB jumpgate + 11 B x SNP entries + 4 B x genome (dense pileup)
    # + the Bloom filters: ~19 GB at S1 size, ~62 GB at GRCh38 size; the index files themselves sit in the page cache once
    big = workload != "s1" and args.scale >= 0.5
    per_proc_gb, files_gb = (62.0, 46.0) if big else (19.0, 2.5)
    if workload != "s1":
        why = None
        if not have_gpu:
            why = "no GPU to build the GRCh38-shaped index with"
        elif not orc.have_ref():
            why = "oracle/_ref/vargeno is not built"
        elif big and mem_available_gb() < 2 * files_gb + per_proc_gb + 16:
            why = "%.0f GB of host memory available; image + files + one reference process need ~%.0f GB" % (mem_available_gb(), 2 * files_gb + per_proc_gb + 16)
        if why:
            fallback, workload, big = why, "s1", False
            per_proc_gb, files_gb = 19.0, 2.5

    def make_inputs(workload, nproc_cap):
        """index image + reads.  With a GPU on the box they come from the device-side builder (seconds, byte-identical index);
        without one (S1 only), from the numpy tooling.  Neither is part of what is timed."""
        sub, lowq = READ_SETS[workload]
        total = nproc_cap * nb * Bp
        if have_gpu:
            from vargeno_b200.geno import Genotyper
            from vargeno_b200.tools import device_workloads as dw
            with Genotyper(device=0) as g:
                dwl = build_workload(g, workload, args.scale, keep_host=True)
                out = g.dalloc(total * rec_bytes(L))
                dw.synth_batch(g, dwl, out, total, 0, sub, lowq, LOWQ_CHARS, REC_ID_WIDTH)
                text = g.d2h(out, total * rec_bytes(L))
                return dwl.host_index, text, dwl.name, dwl.index_counts, g.n_sites
        wl = workloads.make_s1(scale=args.scale)
        text = synth.simulate_reads(wl.genome, wl.haps, total, L, seed=wl.seed + 1000, sub_rate=sub, lowq_prob=lowq,
                                    lowq_chars=LOWQ_CHARS, id_width=REC_ID_WIDTH)
        from oracle import oracle as o2
        oo = o2.Oracle(wl.index)
        n_sites = int(oo.sites().size)
        oo.close()
        return wl.index, text, wl.name, {"ref_kmers": int(wl.index.ref.size), "snp_kmers": int(wl.index.snp.size)}, n_sites

    def run_procs(workload, inp, nproc, load_timeout):
        """inp: {"index", "text"}; the index image is dropped as soon as the files are written (the processes need the memory).
        -> (seconds of the K timed steps, None, load seconds) or (None, why it could not run, None)."""
        text = inp["text"]
        base = "/dev/shm" if big_enough("/dev/shm", files_gb + 1) else None
        d = tempfile.mkdtemp(prefix="vg_refarm_", dir=base)
        procs, fds = [], []
        try:
            prefix = os.path.join(d, workload)
            ib.write_index(inp.pop("index"), prefix)
            vcf = os.path.join(d, "snp.vcf")            # only opened after the read loop (src/qv.cc:1628), which this arm never reaches
            open(vcf, "w").write("##fileformat=VCFv4.0\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")
            fifos = []
            for p in range(nproc):
                ff = os.path.join(d, "reads%d.fq" % p)
                os.mkfifo(ff)
                fifos.append(ff)
                procs.append(subprocess.Popen([orc.REF_BIN, "geno", prefix, ff, vcf, os.path.join(d, "out%d.vcf" % p)],
                                              stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True))
            for p in range(nproc):
                fds.append(os.open(fifos[p], os.O_WRONLY))      # blocks until the process opens its FASTQ (after argv parsing)
            # "Processing..." is printed once the index is loaded (src/qv.cc:753)
            ready = [False] * nproc

            def wait_ready(p):
                for line in procs[p].stderr:
                    if line.startswith("Processing"):
                        ready[p] = True
                        return
            ths = [threading.Thread(target=wait_ready, args=(p,), daemon=True) for p in range(nproc)]
            t_load = time.perf_counter()
            for t in ths:
                t.start()
            for t in ths:
                t.join(max(1.0, load_timeout - (time.perf_counter() - t_load)))
            if not all(ready):
                return None, "reference start-up (index load) not finished after %.0f s in %d of %d processes" % (
                    load_timeout, ready.count(False), nproc), None
            load_s = time.perf_counter() - t_load

            def feed(p, s, res):
                t0 = time.perf_counter()
                off = (p * nb + s) * bb
                mv = memoryview(text)[off:off + bb]
                done = 0
                while done < bb:
                    done += os.write(fds[p], mv[done:done + (1 << 20)])
                res[p] = time.perf_counter() - t0

            step_t = []
            for s in range(nb):
                res = [0.0] * nproc
                th = [threading.Thread(target=feed, args=(p, s, res)) for p in range(nproc)]
                t0 = time.perf_counter()
                for t in th:
                    t.start()
                for t in th:
                    t.join()
                step_t.append(time.perf_counter() - t0)
            return sum(step_t[W:]), None, load_s
        finally:
            for fd in fds:
                try:
                    os.close(fd)
                except OSError:
                    pass
            for pr in procs:
                pr.kill()
            shutil.rmtree(d, ignore_errors=True)

    def plan_nproc():
        avail = mem_available_gb()
        # one process per core that fits beside the index files (page cache / tmpfs), 8 GB for this process and its read set, and
        # a margin of 5 % of the box (at least 10 GB): the per-process figure is an estimate, and a box driven out of memory is
        # worse than one process fewer
        n = int((avail - files_gb - 8 - max(10.0, 0.05 * avail)) // per_proc_gb)
        n = max(1, min(os.cpu_count() or 1, n))
        return args.ref_procs or n

    use_ref = orc.have_ref() and mem_available_gb() > 40
    dt = None
    load_s = None
    if use_ref:
        # the number of processes is planned before the inputs exist (the read set is sized by it); the image copied back from
        # the GPU is dropped as soon as the files are written, so only the files (page cache / tmpfs) and the processes count
        nproc = plan_nproc()
        index, text, name, counts, n_sites = make_inputs(workload, nproc)
        inp = {"index": index, "text": text}
        del index, text
        dt, why, load_s = run_procs(workload, inp, nproc, args.ref_load_timeout)
        if dt is None and workload != "s1":
            fallback, workload, big = why, "s1", False
            per_proc_gb, files_gb = 19.0, 2.5
            inp.clear()
            nproc = plan_nproc()
            index, text, name, counts, n_sites = make_inputs(workload, nproc)
            inp = {"index": index, "text": text}
            del index, text
            dt, why, load_s = run_procs(workload, inp, nproc, args.ref_load_timeout)
        if dt is None:
            use_ref = False
    if not use_ref:
        # the oracle port, one thread (the compiled reference is absent, would not fit in RAM or did not start)
        if workload != "s1":
            fallback, workload = fallback or "the compiled reference cannot run here", "s1"
        index, text, name, counts, n_sites = make_inputs(workload, 1)
        o = orc.Oracle(index)
        times = []
        for s in range(nb):
            t0 = time.perf_counter()
            o.process_fastq(text[s * bb:(s + 1) * bb], want_results=False)
            times.append(time.perf_counter() - t0)
        dt = sum(times[W:])
        value = K * Bp / dt
        kind, cores, sample = "port", 1, "oracle/liboracle.so, 1 thread, %d reads per step" % Bp
    else:
        value = K * Bp * nproc / dt
        kind, cores = "reference", nproc
        sample = ("unmodified reference `vargeno geno` (oracle/_ref), %d processes x 1 thread (the reference is single-threaded; "
                  "one process per core that fits in RAM at ~%.0f GB each), index loaded before timing (%.0f s), %d reads per process per step "
                  "pushed through a FIFO (time = writer completion, pipe slack 64 KiB)" % (nproc, per_proc_gb, load_s or 0.0, Bp))
    if fallback:
        open(FALLBACK_MARK, "w").write(fallback)
    out = {"impl": "reference", "metric": "reads/s", "value": value, "unit": "reads/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
           "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
           "data": "synthetic",
           "config": workload_config(workload, args.scale, name, counts, n_sites),
           "batch": {"reads_per_step": Bp * cores},
           "cpu_baseline": {"value": value, "unit": "reads/s", "cores": cores, "kind": kind, "sample": sample},
           "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    if fallback:
        out["workload_fallback"] = fallback
    emit(out)


def big_enough(path, need_gb):
    try:
        st = os.statvfs(path)
        return st.f_bavail * st.f_frsize / 1e9 >= need_gb
    except OSError:
        return False


_REAL_STDOUT = None


def emit(obj):
    """The one JSON line of this process, on the real stdout."""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def main():
    # Libraries print to fd 1 on their own (NCCL's "NCCL version ..." banner at communicator set-up): everything but the
    # result line goes to stderr, so that stdout carries exactly one JSON line.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the genome / SNP list (tests only)")
    ap.add_argument("--workload", default="s2", choices=["s1", "s2", "s3"],
                    help="s2: GRCh38-shaped WGS reads (BASELINE configs[2], what the metric is quoted on; the default); "
                         "s1: chr22-shaped (configs[1]); s3: high-error stress (configs[3])")
    ap.add_argument("--batch-reads", type=int, default=2_000_000)
    ap.add_argument("--cpu-sample", type=int, default=400_000)
    ap.add_argument("--ref-batch-reads", type=int, default=100_000)
    ap.add_argument("--ref-procs", type=int, default=0)
    ap.add_argument("--ref-load-timeout", type=float, default=540.0,
                    help="seconds the reference processes get to load the index (214 s measured at GRCh38 size; the S1 fallback behind it must still fit the driver's per-run limit)")
    ap.add_argument("--probe-launches", type=int, default=38, help="S4: launches of 2^28 k-mers per probe set (38 = 10^10 k-mers)")
    ap.add_argument("--clock-hold-s", type=float, default=1.0, help="extra seconds of the same load while nvidia-smi samples clocks")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-shapes", action="store_true", help="do not run the S3 / S4 legs after the S2 legs")
    ap.add_argument("--skip-roofline-probe", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed (site counters, calls, step counters) as DIR/<name>.npy, to compare builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed: it does not apply to --impl reference")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
