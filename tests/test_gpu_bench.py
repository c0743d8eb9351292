"""bench.py end to end at a small scale of the default (GRCh38-shaped) workload: the one JSON line must carry what the contract
names, and the full-size parity check it performs against the CPU port (cpu_baseline.parity) must come out green -- the same
code path the driver runs at scale 1."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_line_at_small_scale(tmp_path):
    dump = str(tmp_path / "outputs")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--scale", "0.004", "--steps", "2", "--warmup", "3", "--batch-reads", "20000",
                        "--cpu-sample", "6000", "--probe-launches", "1", "--clock-hold-s", "0", "--dump-outputs", dump],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, p.stdout[-2000:]
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert k in d, k
    assert d["metric"] == "reads/s" and d["n_gpus"] == 1 and d["steps"] == 2 and d["value"] > 0
    assert d["config"]["baseline_config"] == "configs[2]" and "workload" in d["config"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and r["peak"] > 0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["launch_ms"] > 0 and r["algorithmic_bytes_per_launch"] > 0
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 20000 * 316 and e["d2h_bytes_per_step"] > 0
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] == 1 and c["value"] > 0
    assert c["parity"]["parity_checked"] is True and c["parity"]["reads_compared"] == 6000 and c["parity"]["counters_differing"] == []
    assert c["parity_s3"]["parity_checked"] is True and c["parity_s3"]["reads_compared"] == 1500 and c["parity_s3"]["counters_differing"] == []
    assert d["gpu_launches"] > 0
    assert set(d["shapes"]) == {"s3", "s4"} and d["shapes"]["s3"]["value"] > 0
    # --dump-outputs: float arrays of what the timed leg computed; the step counters cover exactly the --steps timed steps
    o = d["dump_outputs"]
    got = {f[:-4]: np.load(os.path.join(dump, f)) for f in sorted(os.listdir(dump))}
    assert sorted(got) == ["alt_cnt", "conf", "counters", "gt", "ref_cnt", "site_index"] and o["files"] == sorted(f + ".npy" for f in got)
    assert all(a.dtype in (np.float32, np.float64) for a in got.values()) and sum(a.nbytes for a in got.values()) <= 64 << 20
    n = min(d["config"]["snp_sites"], 1 << 20)
    assert o["sites"] == n and all(got[k].shape == (n,) for k in ("site_index", "ref_cnt", "alt_cnt", "gt", "conf"))
    counters = dict(zip(o["counters"], got["counters"]))
    assert counters["reads"] == 2 * 20000 and counters["placed"] > 0
    assert np.count_nonzero(got["ref_cnt"] + got["alt_cnt"]) > 0 and np.isin(got["gt"], [0, 1, 2, 3]).all()
