"""bench.py's command line: the JSON contract of the reference arm's line (CPU alone) and the outputs --dump-outputs
writes (the reference arm here, the GPU arm on a small run)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import synth_ref
import util
from oracle import oracle

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*extra):
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--cpu-grid", "24", "--cpu-scale", "12"] + list(extra), capture_output=True, text=True, timeout=300,
                       cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "stdout must carry exactly one JSON line"
    return json.loads(lines[0])


def test_reference_arm_line_has_the_contract_keys():
    d = run_bench()
    assert d["impl"] == "reference" and d["metric"] == "spmv_effective_bandwidth" and d["unit"] == "GB/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] == 1 and cb["value"] == d["value"] and cb["sample"]
    assert cb["all_cores"]["kind"] == "port" and cb["all_cores"]["cores"] >= 1 and cb["all_cores"]["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None


def test_reference_arm_other_workloads():
    for extra in (["--workload", "rmat"], ["--format", "tjds"], ["--workload", "rmat", "--format", "tjds"]):
        d = run_bench(*extra)
        assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1", "--cpu-grid", "10"], capture_output=True, text=True, timeout=120, cwd=REPO, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.parametrize("args,message", [
    (["--steps", "0"], "--steps must be at least 1"),
    (["--secondary-steps", "0"], "--secondary-steps must be at least 1"),
    (["--cpu-iters", "0"], "--cpu-iters must be at least 1"),
    (["--warmup", "-1"], "--warmup must not be negative"),
    (["--format", "tjds", "--gpus", "2", "--exchange", "none", "--dump-outputs", "out"], "needs an exchange"),
])
def test_bad_arguments_are_refused(args, message):
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference"] + args,
                       capture_output=True, text=True, timeout=120, cwd=REPO)
    assert r.returncode == 2 and message in r.stderr


def test_reference_arm_dumps_its_output(tmp_path):
    run_bench("--dump-outputs", str(tmp_path))
    assert os.listdir(tmp_path) == ["y.npy"]
    y = np.load(tmp_path / "y.npy")
    # the 24^3 stencil with {26, -1} values times x = ones: 27 - (entries in the row), exactly
    assert y.dtype == np.float64 and np.array_equal(y, 27.0 - synth_ref.stencil27_row_counts(24, 24, 24))


def test_dump_rows_are_all_rows_or_a_fixed_sample():
    assert np.array_equal(bench.dump_rows(1000, 1000), np.arange(1000))
    s = bench.dump_rows(50_000_000, 1 << 16)
    assert np.array_equal(s, bench.dump_rows(50_000_000, 1 << 16)), "the sample is the same from run to run"
    assert 0.95 * (1 << 16) < len(s) <= 1 << 16 and np.all(np.diff(s) > 0) and 0 <= s[0] and s[-1] < 50_000_000
    assert bench.output_name("stencil 369^3 TJDS deterministic_fast") == "y_stencil_369_3_tjds_deterministic_fast"


@pytest.mark.gpu
@pytest.mark.parametrize("limits", [None, (5000, 1000)], ids=["all_rows", "sampled_rows"])
def test_dump_outputs_are_the_products_of_the_timed_steps(tmp_path, limits):
    """--dump-outputs on a small GPU run: one y per timed configuration, each the product of the seeded matrix and the
    seeded x of the timed steps (not the x = ones of the closed-form check that runs after them), within 1e-12.
    `limits` lowers the row budgets below the lengths of the outputs, so the sampled rows are checked too."""
    g, scale = 24, 12
    argv = ["--steps", "3", "--warmup", "1", "--grid", str(g), "--secondary-scale", str(scale), "--secondary-steps", "2",
            "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)]
    if limits is None:
        cmd = [sys.executable, os.path.join(REPO, "bench.py")] + argv
        limits = (bench.DUMP_ROWS, bench.DUMP_ROWS_SECONDARY)
    else:
        cmd = [sys.executable, "-c", "import sys, bench; bench.DUMP_ROWS, bench.DUMP_ROWS_SECONDARY = %d, %d; "
               "sys.argv[0] = 'bench.py'; bench.main()" % limits] + argv
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=REPO)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads(r.stdout)
    assert d["steps"] == 3 and len(d["secondary"]) == 7
    tjds = ("atomic", "deterministic", "deterministic_fast")
    want = {"y": "stencil"}
    want.update({"y_stencil_%d_3_tjds_%s" % (g, v): "stencil" for v in tjds})
    want.update({"y_r_mat_scale_%d_%s" % (scale, a): "rmat" for a in ["csr"] + ["tjds_" + v for v in tjds]})
    assert sorted(os.listdir(tmp_path)) == sorted(name + ".npy" for name in want)
    mats = {"stencil": (g ** 3, synth_ref.stencil27(g, g, g)), "rmat": (1 << scale, synth_ref.rmat(scale, 16 << scale, seed=42))}
    y_ref = {k: oracle.csr_mult(*oracle.csr_build(coo, n, n), synth_ref.vector(n, 12345)) for k, (n, coo) in mats.items()}
    for name, mat in want.items():
        rows = bench.dump_rows(mats[mat][0], limits[0] if name == "y" else limits[1])
        y = np.load(tmp_path / (name + ".npy"))
        assert y.dtype == np.float64 and len(y) == len(rows), name
        assert util.rel_l2(y, y_ref[mat][rows]) <= 1e-12, name
