"""The bench.py contract, checked on the CPU: the reference
arm (`--impl reference`: the UNMODIFIED reference over the BEAGLE-equivalent CPU
kernels when oracle/_ref is built, else the oracle port) prints exactly one JSON
line on stdout with the agreed keys, and the last committed line of our own arm
(profiles/r02_bench.json) carries roofline / e2e / cpu_baseline and the config legs as specified.
On the device: --dump-outputs writes what the timed path returns."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
             "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def test_reference_arm_prints_one_contract_line():
    done = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                           "--warmup", "0", "--trees", "8", "--patterns", "2000"], capture_output=True, text=True,
                          timeout=600, cwd=ROOT)
    assert done.returncode == 0, done.stderr[-2000:]
    lines = [line for line in done.stdout.splitlines() if line.strip()]
    assert len(lines) == 1, done.stdout
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and BASE_KEYS <= set(line)
    assert line["metric"] == "tree logL+branch-gradient evals/sec" and line["unit"] == "evals/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] and "sample" in line["cpu_baseline"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_committed_bench_line_of_our_arm():
    line = json.loads(open(os.path.join(ROOT, "profiles", "r02_bench.json")).read())
    assert BASE_KEYS | {"clocks", "roofline"} <= set(line) and "impl" not in line
    assert line["dtype"] == "f64" and line["data"] == "synthetic" and line["vs_baseline"] is None
    assert line["scaling"] == "strong" and line["config"]["trees"] == 1024
    roofline = line["roofline"]
    assert roofline["bound"] == "hbm" and roofline["unit"] == "GB/s"
    # frac is a utilisation: measured DRAM bytes of the launch / kernel time / measured peak, never above 1
    assert roofline["traffic"] is not None and "measured in this run" in roofline["traffic_source"]
    assert abs(roofline["achieved"] - roofline["traffic"] / (roofline["kernel_ms"] * 1e-3) / 1e9) < 1e-6 * roofline["achieved"]
    assert abs(roofline["frac"] - roofline["achieved"] / roofline["peak"]) < 1e-9 and 0 < roofline["frac"] <= 1
    # the algorithmic-bytes equivalent is reported separately: (10 n - 14) x 32 C P per tree (SURVEY.md 8d)
    config = line["config"]
    per_tree = (10 * config["taxa"] - 14) * 32 * config["categories"] * config["patterns"]
    assert roofline["algorithmic_bytes_per_launch"] == per_tree * config["trees_per_gpu"]
    assert roofline["traffic"] < roofline["algorithmic_bytes_per_launch"]
    assert abs(roofline["algorithmic_equiv_frac"] -
               roofline["algorithmic_bytes_per_launch"] / (roofline["kernel_ms"] * 1e-3) / 1e9 / roofline["peak"]) < 1e-9
    assert line["gpu_launches"] > 0 and line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert line["e2e"]["value"] <= line["value"] * 1.02  # host buffers + copies cannot beat the resident run
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    # the other BASELINE.json configs ride on the same line
    assert "configs[4]" in line["config5"]["workload"] and line["config5"]["value"] > 0
    assert line["config5"]["oracle_check"]["logl_rel_err"] < 1e-10
    assert line["config5"]["oracle_check"]["gradient_rel_err"] < 1e-8
    cases = line["small_problem"]["cases"]
    assert {c["trees"] for c in cases} == {10, 100} and all(c["gpu_us_per_call"] > 0 for c in cases)
    assert line["e2e_full_phylo_gradients"]["value"] > 0


def test_steps_set_the_number_of_timed_steps():
    done = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                          text=True, timeout=600, cwd=ROOT)
    assert done.returncode != 0 and "--steps must be at least 1" in done.stderr


def test_dumped_outputs_are_a_fixed_sample_under_the_size_limit(tmp_path, monkeypatch):
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 200_000)
    logl = np.arange(1000.0)
    grad = np.arange(1000.0)[:, None] * np.ones((1, 39))
    for directory in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(directory), log_likelihoods=logl, branch_gradients=grad)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 200_000
    index = np.load(tmp_path / "a" / "tree_index.npy")
    assert np.all(np.diff(index) > 0) and len(index) > 500
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "log_likelihoods.npy"), index)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "branch_gradients.npy"), grad[index.astype(int)])
    for name in ("tree_index", "log_likelihoods", "branch_gradients"):
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy"))


@pytest.mark.gpu
def test_dumped_outputs_are_what_the_timed_path_returns(tmp_path):
    """--dump-outputs holds the last timed step's results; the same staged run made here
    on the same seeded inputs gives them again."""
    import argparse
    import numpy as np
    import bench
    import libsbn_b200 as sbn
    from libsbn_b200 import _capi
    size = argparse.Namespace(taxa=12, patterns=2000, trees=8)
    done = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--quick",
                           "--no-cpu-baseline", "--no-traffic-probe", "--taxa", "12", "--patterns", "2000",
                           "--trees", "8", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                          timeout=600, cwd=ROOT)
    assert done.returncode == 0, done.stderr[-2000:]
    states, weights, parent_ids, lengths, params = bench.workload(size)
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", "weibull+4", "none"), states, weights, 0)
    staged = engine.stage(sbn.TreeBatch(parent_ids, lengths), params)
    staged.run(_capi.MODE_BRANCH_GRADIENT, True)
    want = dict(zip(("log_likelihoods", "branch_gradients", "rate_gradients"), staged.fetch(gradients=True)))
    assert sorted(os.listdir(tmp_path)) == sorted(name + ".npy" for name in want)
    for name, value in want.items():
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == np.float64 and got.shape == value.shape
        np.testing.assert_allclose(got, value, rtol=1e-12, atol=1e-300)
