"""`bench.py --impl reference` (the reference's CPU operators timed on host cores) needs no GPU, so its contract is
checked here: one JSON line with the shared keys, `impl: reference`, a `cpu_baseline` describing the run and an `e2e`
equal to the line's own value with no host<->device bytes; under torchrun only rank 0 works and prints.  Where the
reference's operators were not built (oracle/_ref), the arm times the C restatement instead (`kind: port`)."""
import json
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _json_lines(text: str):
    out = []
    for ln in text.splitlines():
        ln = ln.strip()
        if ln.startswith("{") and ln.endswith("}"):
            try:
                out.append(json.loads(ln))
            except json.JSONDecodeError:
                pass
    return out


def _check(line):
    assert line["impl"] == "reference"
    assert line["metric"].startswith("decode tokens/sec") and line["unit"] == "tokens/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["ms_per_step"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == line["value"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"] and "where" not in line["config"]
    # the protocols of BASELINE.md 3.2: stock (64 threads, unbound), bound to cores, tuned to the usable physical cores
    assert cb["protocol"] in cb["protocols"] and "stock" in cb["protocols"] and "stock_pinned" in cb["protocols"]
    assert cb["physical_cores_usable"] >= 1 and cb["threads"] >= 1 and cb["host"]["logical_cpus"] >= 1
    best = min(v["ms_per_layer"] for v in cb["protocols"].values() if "ms_per_layer" in v)
    assert abs(best - cb["ms_per_layer"]) < 1e-9


@pytest.mark.timeout(600)
def test_reference_arm_single():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, cwd=ROOT, timeout=580)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1, r.stdout[-2000:]
    _check(lines[0])
    assert lines[0]["n_gpus"] == 1 and lines[0]["steps"] == 1 and lines[0]["warmup"] == 1


@pytest.mark.timeout(600)
def test_reference_arm_under_torchrun_rank0_only():
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", str(_free_port()), os.path.join(ROOT, "bench.py"), "--gpus", "2", "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--P", "6000", "--M", "8192"],   # a small context: this test is about who runs and prints
                       capture_output=True, text=True, cwd=ROOT, timeout=580, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1, r.stdout[-2000:]      # rank 1 exits 0 without work or output
    _check(lines[0])
    assert lines[0]["n_gpus"] == 2


def test_tracked_bench_lines_keep_the_contract():
    """The bench lines committed under profiles/ (what DESIGN.md quotes) carry every key of the bench.py contract and their
    derived numbers are consistent with each other."""
    BASE = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    for name, full in [("r2_bench_line.json", True), ("r2_bench_line_final_kernel.json", False), ("r2_bench_c3_b8.json", False),
                       ("r2_bench_c4_prolong.json", False)]:
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            pytest.skip(f"{name} not tracked")
        d = _json_lines(open(path).read())[-1]
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                  "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"):
            assert k in d, (name, k)
        assert d["unit"] == "tokens/s" and d["higher_is_better"] is True and d["n_gpus"] == 1 and d["warmup"] >= 3
        assert d["gpu_launches"] > 0 and d["data"].startswith("synthetic")
        assert abs(d["value"] - 1e3 / d["ms_per_step"] * d["config"].get("global_batch", 1)) / d["value"] < 1e-6
        e2e = d["e2e"]
        assert 0 < e2e["value"] <= d["value"] * 1.001 and e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0
        r = d["roofline"]
        assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        assert abs(r["achieved"] - r["bytes_per_launch"] / (r["us_per_launch"] * 1e-6) / 1e9) / r["achieved"] < 1e-6
        assert not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"]))
        if full:
            assert BASE["metric"].startswith(d["metric"])   # BASELINE.json names the metric (+ the roofline it wants beside it)
            cb = d["cpu_baseline"]
            assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["sample"] and cb["value"] > 0
            assert r["traffic"] is None or r["traffic"] >= 0.9 * r["bytes_per_launch"]
