"""bench.py's CPU legs (the `cpu_baseline` block and `--impl reference`): the committed strategy-state fixture
they start from, and the line the reference arm prints.  No GPU needed."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_bench_state_fixture_is_the_converged_regime():
    """tests/golden/bench_state_gen30.npz (tools/make_bench_fixture.py): offspring drawn around it with the twin
    run the full 500 steps, i.e. the CPU legs are timed in the regime of the GPU arm's timed generations."""
    import bench
    from oracle import twin
    st = bench.bench_state()
    assert st["mu"].shape == (bench.D,) and st["mu"].dtype == np.float32 and st["t"] == 30
    assert abs(st["sigma"] - 0.2 * 0.9999 ** 30) < 1e-15
    fit, steps = twin.population_cartpole(st["mu"][None], sigma=st["sigma"], seed=0, gen=30, group=bench.P_DEFAULT,
                                          n_head=1, n=64, E=bench.E_DEFAULT, nthreads=2)
    assert steps.sum() / (64 * bench.E_DEFAULT) > 490
    hist = np.load(bench.STATE_FIXTURE)["history"]
    assert hist.shape == (30, 3) and hist[-1, 2] > 499.9 and hist[0, 2] < 25


def test_reference_generation_port_from_state():
    """One tiny generation of the reference-path port from the fixture state: 2 offspring (mu itself and one
    perturbation), every episode 500 steps."""
    import bench
    steps, dt = bench.cpu_reference_generation(2, 1, 7, eval_ep_num=1, state=bench.bench_state())
    assert steps == 2 * 500 and dt > 0


def test_dump_outputs_writes_float_arrays_and_samples_above_the_cap(tmp_path, monkeypatch):
    """--dump-outputs: float32 stays float32, every other dtype becomes float64; above the size cap the per-offspring arrays
    are cut to the same seeded sample of offspring on every call, and their ids are written too."""
    import torch
    import bench
    P, D = 5000, 226
    off = {"fitness": torch.arange(P, dtype=torch.float64) * 0.5, "rank_order": torch.arange(P - 1, -1, -1, dtype=torch.int32)}
    par = {"mu": torch.linspace(-1, 1, D, dtype=torch.float32)}
    bench.dump_outputs(str(tmp_path / "full"), off, par)
    got = {p.stem: np.load(p) for p in (tmp_path / "full").iterdir()}
    assert sorted(got) == ["fitness", "mu", "rank_order"]
    assert got["mu"].dtype == np.float32 and np.array_equal(got["mu"], par["mu"].numpy())
    assert got["rank_order"].dtype == np.float64 and np.array_equal(got["rank_order"], np.arange(P - 1, -1, -1))
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", D * 4 + 1000 * 24)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), off, par)
    a = {p.stem: np.load(p) for p in (tmp_path / "a").iterdir()}
    ids = a["offspring_ids"].astype(np.int64)
    assert len(ids) == 1000 and np.all(np.diff(ids) > 0) and sum(x.nbytes for x in a.values()) <= bench.DUMP_LIMIT_BYTES
    assert np.array_equal(a["fitness"], ids * 0.5) and np.array_equal(a["rank_order"], P - 1 - ids)
    assert all(np.array_equal(a[k], np.load(tmp_path / "b" / (k + ".npy"))) for k in a)


def test_reference_arm_line_keys():
    env = dict(os.environ, RANK="0")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["gpu_launches"] == 0 and line["higher_is_better"] is True
    assert line["unit"] == "env-steps/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == (os.cpu_count() or 1)
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["config"]["population"] == 65536


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""
