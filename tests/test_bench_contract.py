"""CPU: the JSON lines bench.py prints carry every key of the driver contract (both arms). The GPU arm is exercised through
tests/emu/bench_dryrun.py (emulation build, stubbed torch.cuda streams / events: control flow and JSON assembly only -- the
numbers of a dry run mean nothing); the reference arm runs for real on a tiny mesh."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _last_json(out):
    lines = [ln for ln in out.strip().splitlines() if ln.startswith("{")]
    assert lines, out[-2000:]
    return json.loads(lines[-1])


def test_gpu_arm_json_line_has_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "bench_dryrun.py")], capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, B2P_BENCH_EXPERIMENTS="0"), cwd=ROOT)
    d = _last_json(r.stdout + r.stderr)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["unit"] == "MDoF/s" and d["dtype"] == "f64" and d["scaling"] == "weak" and d["vs_baseline"] is None and d["n_gpus"] == 1
    assert "workload" in d["config"] and "model" not in d["config"]
    assert set(("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")) <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
    assert set(("bound", "achieved", "peak", "unit", "frac", "traffic")) <= set(d["roofline"]) and d["roofline"]["bound"] == "hbm"
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] in ("port", "reference")
    assert d["gpu_launches"] > 0


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--n", "4"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    d = _last_json(r.stdout)
    assert d["impl"] == "reference" and d["unit"] == "MDoF/s" and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1


def test_reference_arm_runs_on_rank_zero_only():
    """Under torchrun (N > 1) rank 0 alone times the CPU implementation; the other ranks exit 0 without work or output."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--n", "4"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2"))
    assert r.returncode == 0 and not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_dumped_outputs_of_both_arms_agree(tmp_path):
    """--dump-outputs: the GPU arm (dry run on the emulation build) and the reference arm write y = A x of their last timed
    step for the same seeded x on the same mesh, and the two agree."""
    gpu, ref = tmp_path / "gpu", tmp_path / "ref"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "bench_dryrun.py"), "--no-cpu-baseline", "--dump-outputs", str(gpu)],
                       capture_output=True, text=True, timeout=900, env=dict(os.environ, B2P_BENCH_EXPERIMENTS="0"), cwd=ROOT)
    assert _last_json(r.stdout + r.stderr)["steps"] == 3
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n", "3", "--steps", "2", "--warmup", "1",
                        "--dump-outputs", str(ref)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert _last_json(r.stdout)["steps"] == 2
    yg, yr = np.load(gpu / "y.npy"), np.load(ref / "y.npy")
    assert yg.dtype == yr.dtype == np.float64 and yg.shape == yr.shape and yg.size > 0
    assert np.abs(yg - yr).max() <= 1e-12 * np.abs(yr).max()


def test_experiment_lines_precede_the_headline_line():
    """Every side measurement is its own short JSON line {"experiment": ...} and the headline is the LAST line, so that no
    experiment can fall off a log tail and no headline key can be pushed out by them (VERDICT r01, weak #9)."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "bench_dryrun.py")], capture_output=True, text=True, timeout=1500,
                       env=dict(os.environ, B2P_BENCH_EXPERIMENTS="1", B2P_BENCH_EXPERIMENT_BUDGET_S="600"), cwd=ROOT)
    lines = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) >= 4, r.stdout[-2000:] + r.stderr[-2000:]
    assert "metric" in lines[-1] and "experiment" not in lines[-1] and "experiments" not in lines[-1]
    names = [ln["experiment"] for ln in lines[:-1]]
    assert all("experiment" in ln for ln in lines[:-1])
    assert "matrix_coefficient_warped_mesh" in names and "round1_kernel_nd_hex_apply4" in names
    ok = [ln for ln in lines[:-1] if ln["experiment"] == "matrix_coefficient_warped_mesh"][0]
    assert "failed" not in ok and ok["kernel"] == "nd_hex_apply6_kernel", ok
    assert max(len(json.dumps(ln)) for ln in lines) < 4000
