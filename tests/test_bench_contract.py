"""The driver-facing contract of bench.py: ONE JSON line on stdout with the agreed keys, for the
reference arm (CPU, runs everywhere) and for the GPU arm."""

import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
             "scaling", "vs_baseline", "dtype", "data", "config", "e2e"}


def _run(args, timeout):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, timeout=timeout,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "stdout must carry exactly one line, got %d" % len(lines)
    return json.loads(lines[0])


def _checkReferenceLine(d, kind):
    assert BASE_KEYS <= set(d)
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["metric"] == "chain-iterations/sec" and d["value"] > 0
    assert d["config"]["workload"].startswith("C3")
    cb = d["cpu_baseline"]
    assert cb["kind"] == kind and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_port_prints_one_json_line_with_the_contract_keys():
    """--impl reference on the oracle port (what runs when baseline/_ref is not staged)."""
    d = _run(["--impl", "reference", "--port", "--steps", "1", "--warmup", "0", "--port-iters", "3"], 600)
    _checkReferenceLine(d, "port")


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "baseline", "_ref", "posteriorSampling.py")),
                    reason="baseline/_ref is staged by __graft_entry__.build() where /root/reference exists")
def test_reference_arm_times_the_unmodified_reference():
    """--impl reference runs the unmodified reference's samplePosterior (own process, own modules) on a slice
    of the groups and scales the rate to the full shape; the calibration runs are skipped here (minutes)."""
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-groups", "16", "--no-calibration"], 600)
    _checkReferenceLine(d, "reference")
    assert "unmodified reference" in d["cpu_baseline"]["sample"] and "16/1024" in d["cpu_baseline"]["sample"]
    # one chain-iteration of the reference at this shape takes seconds, not milliseconds
    assert d["value"] / d["cpu_baseline"]["cores"] < 5.0


def test_reference_runner_imports_the_reference_not_the_product():
    """baseline/run_reference.py must time /root/reference's module, never the product module of the same name."""
    src = open(os.path.join(ROOT, "baseline", "run_reference.py")).read()
    assert "assert os.path.dirname(os.path.abspath(reference.__file__)) == REF" in src
    assert "mcmc-for-nested-data_b200" not in src


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun (N > 1) rank 0 alone runs the reference arm; the other ranks exit 0 without work."""
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], cwd=ROOT,
                       timeout=120, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_gpu_arm_prints_one_json_line_with_roofline_and_e2e():
    d = _run(["--steps", "4", "--warmup", "3", "--no-cpu-baseline", "--full-iters", "400", "--full-samples", "100"], 900)
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["dtype"] == "f32" and d["data"] == "synthetic" and d["value"] > 1e5
    assert d["gpu_launches"] > 0
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    f = d["full_run"]
    assert f["iterations"] == 400 and f["retained_rows"] == 100 and f["diagnostics"]["keys"] == 9234
    assert f["diagnostics"]["min_ess"] > 0 and f["min_ess_per_s"] > 0
    assert d["diagnostics"]["rows"] >= 6 and d["c4_single_gpu"]["chains"] == 16384 and d["c5_none"]["roofline"]["bound"] == "mufu"
    r = d["roofline"]
    assert r["bound"] in ("tensor", "fp32", "mufu") and r["unit"] in ("TFLOP/s", "Gop/s")
    assert 0 < r["frac"] < 1 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step_the_same_way_twice(tmp_path):
    """--dump-outputs: the rows the last timed step retained and the chain state it left, float32 / float64,
    64 MB at most (a sample of the 1,024 chains at config 3), and identical from two runs with the same arguments."""
    import numpy
    args = ["--steps", "2", "--warmup", "1", "--no-full-run", "--no-sub-records", "--no-cpu-baseline"]
    dumps = []
    for k in range(2):
        out = tmp_path / str(k)
        _run(args + ["--dump-outputs", str(out)], 600)
        dumps.append(dict((f[:-4], numpy.load(str(out / f))) for f in os.listdir(str(out))))
    a, b = dumps
    assert set(a) == set(b) == {"samples", "theta", "scale", "lprior", "ll", "mu", "sigma2"}
    assert sum(v.nbytes for v in a.values()) <= 64e6
    nC = a["theta"].shape[2]
    assert 0 < nC < 1024 and a["theta"].shape == (9, 1024, nC) and a["ll"].shape == (1024, nC)
    assert a["samples"].shape == (5, 9 * 1026, nC) and a["mu"].shape == a["sigma2"].shape == (9, nC)   # iterations 100..140
    for name in a:
        assert a[name].dtype in (numpy.float32, numpy.float64), name
        numpy.testing.assert_array_equal(a[name], b[name], err_msg=name)
