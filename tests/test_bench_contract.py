"""The bench line contract (driver-facing): the committed record lines under profiles/ carry every key the
contract names, with consistent values; `bench.py` parses its flags without a GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _line(name):
    with open(os.path.join(ROOT, "profiles", name)) as f:
        return json.loads(f.read().strip().splitlines()[-1])


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_record_line_has_the_contract_keys(n):
    d = _line(f"r02_bench_n{n}.json")
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks", "parity"):
        assert key in d, key
    assert d["n_gpus"] == n and d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["metric"] == "mash.Sketch Gbases/s" and d["unit"] == "Gbases/s" and d["data"] == "synthetic" and d["dtype"] == "u32"
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["warmup"] >= 3 and d["gpu_launches"] >= d["steps"] > 0
    # value is the whole-job aggregate: units of all ranks / max-over-ranks time
    reads = d["config"]["reads_per_gpu"] * d["config"]["read_len"] * n
    assert abs(d["value"] - reads / d["ms_per_step"] / 1e6) / d["value"] < 1e-6
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or r["traffic"] > 0
    e = d["e2e"]
    assert e["unit"] == "Gbases/s" and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < d["value"]
    c = d["clocks"]
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert all(d["parity"].values())
    if n == 1:
        cb = d["cpu_baseline"]
        assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and cb["sample"]
        assert all(s["parity_vs_oracle"] for s in d["secondary"])
    else:
        assert d["pipeline"]["parity_all_green"] is True


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_reference_arm_line(n):
    d = _line(f"r02_bench_ref_n{n}.json")
    assert d["impl"] == "reference" and d["metric"] == "mash.Sketch Gbases/s" and d["unit"] == "Gbases/s"
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]


def test_bench_cli_parses_without_a_gpu():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dump-outputs"):
        assert flag in out.stdout


@pytest.mark.gpu
def test_dump_outputs_repeat_and_match_the_oracle(tmp_path, oracle):
    """--dump-outputs: the same files, bit for bit, from two runs with different --steps; --steps sets the timed
    launches; every checked row is the oracle's sketch of the read its index names."""
    import numpy as np

    from poly_b200 import synth

    per_step = []
    for steps in (2, 3):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                              "--reads", "100000", "--no-cpu", "--no-e2e", "--no-secondary", "--dump-outputs", str(tmp_path / str(steps))],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-3000:]
        d = json.loads(out.stdout.strip().splitlines()[-1])
        assert d["steps"] == steps and d["gpu_launches"] % steps == 0 and all(d["parity"].values())
        per_step.append(d["gpu_launches"] // steps)
    assert per_step[0] == per_step[1] > 0
    names = sorted(p.name for p in (tmp_path / "2").iterdir())
    assert names == ["read_index.npy", "sketches.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "2").iterdir()) <= 64 << 20
    for name in names:
        assert np.array_equal(np.load(tmp_path / "2" / name), np.load(tmp_path / "3" / name))
    sk, idx = np.load(tmp_path / "2" / "sketches.npy"), np.load(tmp_path / "2" / "read_index.npy")
    assert sk.dtype == idx.dtype == np.float64 and sk.shape == (32768, 129) and idx.shape == (32768,)
    assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < 100000
    for row in range(0, len(idx), 1024):
        read = synth.independent_reads(1, 150, first_read=int(idx[row]))
        rc, want = oracle.sketch_batch(read, synth.uniform_offsets(1, 150), 21, 1000, variant=1)
        assert rc == 0 and np.array_equal(sk[row], want[0, :129].astype(np.float64)), row


def test_documented_numbers_trace_to_the_record_lines():
    """The round-2 tables of README.md / DESIGN.md quote the committed bench lines (within rounding)."""
    import re

    d1, d8 = _line("r02_bench_n1.json"), _line("r02_bench_n8.json")
    sec = {s["name"]: s for s in d1["secondary"]}
    readme = open(os.path.join(ROOT, "README.md")).read()
    design = open(os.path.join(ROOT, "DESIGN.md")).read()

    def quoted(text, pattern):
        m = re.search(pattern, text)
        assert m, pattern
        return float(m.group(1))

    assert abs(quoted(readme, r"\*\*1\.56 ms / pass = (\d+) Gbases/s\*\*") - d1["value"]) / d1["value"] < 0.01
    assert abs(quoted(readme, r"\*\*(\d+) Gbases/s \(7\.99×\)\*\*") - d8["value"]) / d8["value"] < 0.005
    assert abs(quoted(readme, r"cfg3 \(100 k × 10 kbp, k=31, s=2000\) \| \*\*([\d.]+) ms") - sec["cfg3 sketch (K2)"]["ms"]) < 0.03
    assert abs(quoted(readme, r"\*\*([\d.]+) ms = 6\.45 TCUPS\*\*") - sec["cfg5 Smith-Waterman score (K4)"]["ms"]) < 0.2
    assert abs(quoted(design, r"\| 15\.5 / 30\.1 / 49\.2 / \*\*([\d.]+) Gbases/s\*\*") - d8["e2e"]["value"]) < 0.3
    assert abs(quoted(design, r"0\.656 of HBM peak \| unchanged \(1\.56 ms, (\d+) Gbases/s") - d1["value"]) / d1["value"] < 0.01
    assert abs(d1["roofline"]["frac"] - 0.656) < 0.01
