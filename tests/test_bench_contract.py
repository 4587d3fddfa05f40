"""bench.py contract, CPU side: the reference arm (the CPU restatement of the path, the one other
place that may execute oracle/) prints exactly ONE JSON line with the agreed keys, and importing
bench.py has no side effects on the process' stdout."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_reference_arm_prints_one_json_line():
    # (the default workload, fsi_512_f32, needs ~35 GB of host memory and minutes of CPU: a named small
    # workload with a body exercises the same code)
    env = dict(os.environ, OMP_NUM_THREADS="1")  # as torchrun exports it: the arm must not inherit it
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--workload", "rod_fsi_128x64x64_f32"], capture_output=True, text=True,
                       timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "impl"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "full_timestep_Mcell_updates_per_s"
    assert d["unit"] == "Mcell-updates/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["config"]["workload"] == "rod_fsi_128x64x64_f32" and d["config"]["grid_zyx"] == [64, 64, 128]
    assert d["config"]["lagrangian_points"] > 10000 and d["scaling"] == "strong"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--gpus", "2"], capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_default_workload_is_the_north_star_target():
    sys.path.insert(0, ROOT)
    import bench

    assert bench.DEFAULT_WORKLOAD == "fsi_512_f32"
    grid, flow_type, body, prec = bench.WORKLOADS[bench.DEFAULT_WORKLOAD]
    assert grid == (512, 512, 512) and flow_type == "navier_stokes_with_forcing" and body and prec == "f32"
    w = bench.workload_setup("fsi_256_f32", (256, 256, 256))
    assert w["points"].shape[0] == 3 and w["points"].shape[1] > 30000
    # the CPU arm is bounded: one 512^3 step, a few 128^3 steps
    assert bench.cpu_arm_steps(512 ** 3, 20, 3) == (1, 0)
    assert bench.cpu_arm_steps(128 ** 3, 20, 3) == (20, 1)


def test_importing_bench_leaves_stdout_alone(capfd):
    sys.path.insert(0, ROOT)
    import bench  # noqa: F401

    print("still here")
    out, _ = capfd.readouterr()
    assert "still here" in out


def test_bench_rejects_bad_step_count_and_dump_of_reference_arm():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                           timeout=120)
        assert r.returncode == 2 and r.stdout == "", (extra, r.stderr[-2000:])


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["vortex_ring_128_f32", "rod_fsi_128x64x64_f32"])
def test_dumped_outputs_do_not_depend_on_the_warmup(workload, tmp_path):
    """--dump-outputs: the timed steps start from the initial condition whatever the warm-up, so two runs
    with different --warmup write the same outputs (up to the order of the spreading's float atomics)."""
    import numpy as np
    import torch

    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    dumps = []
    for warmup in (1, 4):
        out = tmp_path / f"warmup{warmup}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", "3",
                            "--warmup", str(warmup), "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
        assert line["steps"] == 3 and line["config"]["workload"] == workload
        dumps.append({p.name: np.load(p) for p in sorted(out.iterdir())})
    names = {"dt.npy", "vorticity_field.npy", "velocity_field.npy", "stream_func_field.npy"}
    if workload.startswith("rod"):
        names |= {"lag_grid_forcing_field.npy", "lag_grid_position_mismatch_field.npy"}
    assert set(dumps[0]) == names == set(dumps[1])
    assert sum(os.path.getsize(tmp_path / "warmup1" / n) for n in names) <= 64_000_000
    for name in names:
        a, b = dumps[0][name], dumps[1][name]
        assert a.dtype in (np.float32, np.float64) and a.shape == b.shape and np.isfinite(a).all(), name
        assert np.abs(a - b).max() <= 1e-5 * np.abs(b).max(), name
    # a grid that fits the budget is written whole; 128^3 is sampled
    n_cells = dumps[0]["vorticity_field.npy"].shape[1]
    assert n_cells == 128 * 64 * 64 if workload.startswith("rod") else 10 ** 6 < n_cells < 128 ** 3
