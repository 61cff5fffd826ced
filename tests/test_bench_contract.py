"""bench.py prints ONE JSON line with the keys the driver's contract names — checked for the
reference arm on CPU and for the B200 arm on a GPU (small workload, few steps)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
             "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "e2e",
             "gpu_launches"}


def run_bench(*args, timeout=600):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args],
                         capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must hold exactly one line: %r" % lines
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "0")
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["value"] > 0 and d["unit"] == "reads/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["flow_value"] == 100  # config 1: F* = M


def test_reference_arm_dumps_outputs(tmp_path):
    d = run_bench("--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "0",
                  "--dump-outputs", str(tmp_path))
    out = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(out) == ["flow_value", "kept_sample", "kept_sample_index", "n_kept"]
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    # solve 0 (seed 12345), whatever the number of host threads: all of config 1's 1M reads
    assert out["flow_value"].tolist() == [d["flow_value"]] == [100]
    assert out["n_kept"].tolist() == [d["n_kept"]] == [out["kept_sample"].sum()]
    assert np.array_equal(out["kept_sample_index"], np.arange(1_000_000))


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--gpus", "2", "--steps", "1", "--warmup", "0"], capture_output=True,
                         text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_b200_arm_line(tmp_path):
    d = run_bench("--workload", "c1", "--steps", "3", "--warmup", "3", "--no-cpu-baseline",
                  "--dump-outputs", str(tmp_path))
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["gpu_launches"] > 0
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3
    e = d["e2e"]
    # the headline end-to-end figure starts from the C ABI's 32-bit host columns and does whatever
    # narrowing it uses inside the timed region; the other encodings are reported next to it
    assert e["encode_in_timed_region"] is True and "uint32 start/end" in e["host_input"]
    assert e["h2d_bytes_per_step"] in (2 * 1_000_000, 8 * 1_000_000)
    assert e["d2h_bytes_per_step"] > 0 and e["value"] > 0
    others = {k for k in d if k.startswith("e2e_")}
    assert "e2e_preencoded" in others and d["e2e_preencoded"]["encode_in_timed_region"] is False
    assert d["e2e_preencoded"]["h2d_bytes_per_step"] == 2 * 1_000_000
    assert ("e2e_u32" in others) != (e["transport"] == "start u32, end u32")
    assert d["result"]["quality"]["kept_over_lower_bound"] < 1.06
    assert d["result"]["bundle_path"] == "histogram in shared memory"
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert d["result"]["fstar"] == d["result"]["flow_value"] == 100
    assert d["config"]["workload"].startswith("c1")
    # --dump-outputs: the last timed step's answer; config 1's 1M reads all fit the sample
    out = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    assert out["kept_per_sample"].tolist() == [d["result"]["n_kept"]] == out["n_kept"].tolist()
    assert np.array_equal(out["kept_sample_index"], np.arange(1_000_000))
    assert out["kept_sample"].sum() == d["result"]["n_kept"] and out["fstar"][0] == 100
    # both arms describe the workload with the same dict (the driver compares them)
    ref = run_bench("--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "0")
    assert ref["config"] == d["config"] and ref["cpu_baseline"]["cores"] >= 1


@pytest.mark.gpu
def test_b200_arm_dumps_a_seeded_sample(O, tmp_path):
    # config 2: 5M pairs through the pair filter, so the pair verdicts are a seeded sample and the
    # kept flags index the reads that passed; both against the oracle on the same seeded input
    d = run_bench("--workload", "c2", "--steps", "2", "--warmup", "3", "--no-cpu-baseline",
                  "--dump-outputs", str(tmp_path))
    out = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    bed, tsv = O.artic_scheme()
    a0, a1 = O.parse_amplicons(bed, tsv)
    s, e, q, l = O.gen_reads_amplicon(12345, 5_000_000, 30_000, a0, a1)
    pp, kept = O.filter_pairs(s, e, q, l, 90, 30, a0, a1)
    pidx = out["pair_pass_sample_index"].astype(np.int64)
    assert 0 < len(pidx) <= 1 << 21 and np.all(np.diff(pidx) > 0) and pidx[-1] < 5_000_000
    assert np.array_equal(out["pair_pass_sample"], pp[pidx])
    mask = np.repeat(pp, 2).astype(bool)
    bm, st = O.sync_solve(s[mask].copy(), e[mask].copy(), [30_000], [0, kept], 100,
                          params=(64, 150, 1, 0, 0, 3))
    assert out["n_filtered"].tolist() == [d["result"]["n_filtered"]] == [kept]
    assert out["kept_per_sample"].tolist() == [d["result"]["n_kept"]] == [st.n_kept]
    idx = out["kept_sample_index"].astype(np.int64)
    assert np.array_equal(out["kept_sample"], O.bitmap_to_mask(bm, kept)[idx])
