"""bench.py's repo arm cannot run without a GPU; its control flow and JSON contract can: tests/bench_dry_run.py runs main() on the
SIMT-emulator build with the CUDA-only torch calls stubbed (timings are meaningless and not checked)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_main_dry_run_prints_the_contract_line():
    from tests.emu import build_emu

    build_emu.build()
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bench_dry_run.py"), "T0", "--steps", "2", "--warmup", "3", "--no-parity",
                        "--no-cpu-baseline", "--ops-calls", "1"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline", "ops"):
        assert k in line, k
    assert line["metric"] == "Navier2D timesteps/sec" and line["unit"] == "steps/s" and line["dtype"] == "f64" and line["n_gpus"] == 1
    assert line["steps"] == 2 and line["warmup"] == 3 and line["gpu_launches"] == 2 * line["run"]["launches_per_step"]
    assert line["e2e_error"] is None and line["e2e"]["h2d_bytes_per_step"] == line["e2e"]["d2h_bytes_per_step"] > 0
    assert line["ops_error"] is None
    assert set(line["ops"]["ms_per_transform"]) == {"forward", "backward"} and set(line["ops"]["ms_per_solve"]) == {"hholtz_adi", "poisson"}
    assert line["ops"]["alg_bytes"]["forward"] == 32.0 * 65 * 65
    for key in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert key in line["roofline"], key


import pytest  # noqa: E402


def test_bench_dump_outputs_hold_the_last_timed_step(tmp_path):
    """--dump-outputs writes the state after the warm-up and the timed steps (3 + 2 from the bench's seeded white noise): the numpy
    oracle stepped as often from the same fields gives the same arrays."""
    import numpy as np

    from oracle import rustpde_oracle as o

    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bench_dry_run.py"), "T0", "--steps", "2", "--warmup", "3", "--no-parity",
                        "--no-cpu-baseline", "--no-ops", "--no-e2e", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    ref = o.Navier2D(65, 65, 1e5, 1.0, 1e-2, 1.0, "rbc")
    for name, seed in (("temp", 1), ("velx", 2), ("vely", 3)):
        f = getattr(ref, name)
        f.v = np.random.default_rng(seed).uniform(-0.1, 0.1, size=(65, 65))
        f.forward()
    for _ in range(5):
        ref.update()
    assert sorted(os.listdir(tmp_path)) == ["pres.npy", "temp.npy", "velx.npy", "vely.npy"]
    for name, want in ref.state().items():
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == np.float64 and got.shape == want.shape, name
        assert np.abs(got - want).max() < 1e-9 * np.abs(want).max(), (name, np.abs(got - want).max() / np.abs(want).max())


def test_dump_outputs_sample_is_fixed_and_within_budget(tmp_path):
    """Arrays above their share of the budget are replaced by the same seeded sample of entries in every run; complex arrays are
    written as [..., 2] = real, imaginary part."""
    import numpy as np

    import bench

    rng = np.random.default_rng(7)
    arrays = {"small": rng.standard_normal((5, 4)), "big": rng.standard_normal((300, 200)),
              "cx": rng.standard_normal((300, 100)) + 1j * rng.standard_normal((300, 100))}
    budget = 3 * (4096 + 8000)
    for d in ("a", "b"):
        bench.dump_outputs(arrays, str(tmp_path / d), budget=budget)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= budget
    for name in arrays:
        first, second = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert first.dtype == np.float64 and np.array_equal(first, second), name
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), arrays["small"])

    def sample(a, k):   # the documented rule: default_rng(0) positions without replacement, ascending
        return a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, k, replace=False))]

    assert np.array_equal(np.load(tmp_path / "a" / "big.npy"), sample(arrays["big"], 1000))
    cx = sample(arrays["cx"], 500)
    assert np.array_equal(np.load(tmp_path / "a" / "cx.npy"), np.stack([cx.real, cx.imag], axis=-1))


@pytest.mark.skipif(os.environ.get("B2_SLOW_TESTS") != "1", reason="opt-in (B2_SLOW_TESTS=1): ~1 min on 2 emulated ranks")
def test_bench_main_dry_run_two_ranks():
    """the N > 1 control flow under torchrun: distributed context, all-reduced timings, identical burst counts on every rank,
    standalone operators on slabs (--ops-multi), rank 0 alone prints"""
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29617", os.path.join(ROOT, "tests", "bench_dry_run.py"), "T0", "--gpus", "2", "--steps", "2", "--warmup", "3",
                        "--no-parity", "--no-cpu-baseline", "--ops-calls", "1", "--ops-multi"], capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["n_gpus"] == 2 and line["ops_error"] is None and line["e2e_error"] is None and line["gpu_launches"] == 2 * line["run"]["launches_per_step"]
