"""CPU: the reference arm of bench.py (the oracle's C engine on the host cores) prints ONE JSON line with the keys the driver
reads; the GPU arm refuses to run without a CUDA device instead of falling back."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    # a wrapper that records which shared libraries the arm maps: it must never load the product library
    code = ("import runpy, sys, os; sys.argv = ['bench.py'] + sys.argv[1:]\n"
            "try:\n    runpy.run_path(os.path.join(%r, 'bench.py'), run_name='__main__')\n"
            "except SystemExit as e:\n    rc = e.code or 0\n"
            "maps = open('/proc/self/maps').read()\n"
            "sys.stderr.write('MAPPED_PRODUCT=%%d MAPPED_ORACLE=%%d\\n' %% ('libgripper_sim_b200' in maps, 'liboracle' in maps))\nsys.exit(rc)\n" % ROOT)
    out = subprocess.run([sys.executable, "-c", code, "--impl", "reference", "--steps", "3", "--warmup", "1", "--preroll", "4", "--cpu-seconds", "2"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert "MAPPED_PRODUCT=0 MAPPED_ORACLE=1" in out.stderr, out.stderr[-2000:]
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["metric"].startswith("env-steps/sec") and "substeps" in d["unit"] and d["value"] > 0 and d["n_gpus"] == 1
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "oracle/engine.c" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("acorn_env")
    # --steps / --warmup are honoured (transitions per environment), and ms_per_step is per transition of the sample: the
    # timed region the driver derives (steps x ms_per_step) is the time actually spent in the timed windows
    assert d["steps"] == 3 and d["warmup"] == 1 and d["preroll"] == 4
    assert "3 timed transitions (after 5 untimed from reset)" in cb["sample"]
    assert 0 < d["steps"] * d["ms_per_step"] / 1e3 < 60
    assert "oracle/mjcf.py" in cb["sample"]


def test_action_tapes():
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    u = np.random.default_rng(0).uniform(-1, 1, (1000, 6))
    a = bench.shape_actions(u.copy(), "contact")  # SURVEY.md §8d cfg5: biased towards +x / close
    assert a[:, 0].min() >= 0.2 and a[:, 0].max() <= 1.0 and a[:, 5].max() <= 0.0 and a[:, 5].min() >= -1.0 and np.abs(a[:, 1:5]).max() <= 0.3
    np.testing.assert_array_equal(bench.shape_actions(u.copy(), "uniform"), u)


def test_dump_outputs_writes_float32_samples_of_the_last_step(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import types
    import numpy as np
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_ROWS", 100)
    N, g = 900, torch.Generator().manual_seed(0)
    sim = types.SimpleNamespace(num_envs=N, device=torch.device("cpu"), reward=torch.rand(N, generator=g), done=(torch.arange(N) % 3 == 0).to(torch.uint8),
                                obs=torch.randint(0, 256, (N, 5, 64, 64), generator=g, dtype=torch.uint8),
                                terminal_obs=torch.randint(1, 256, (N, 5, 64, 64), generator=g, dtype=torch.uint8),
                                achieved_goal=torch.rand(N, 2, generator=g), desired_goal=torch.rand(N, 2, generator=g), info=torch.rand(N, 40, generator=g))
    action = torch.rand(N, 6, generator=g)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), sim, action)
    names = ["achieved_goal", "action", "desired_goal", "done", "info", "obs", "reward", "terminal_obs", "terminal_obs_env"]
    assert sorted(p.stem for p in (tmp_path / "a").iterdir()) == names
    out = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in names}
    for n in names:
        assert out[n].dtype == (np.float64 if n == "terminal_obs_env" else np.float32)
        np.testing.assert_array_equal(out[n], np.load(tmp_path / "b" / (n + ".npy")))  # the sample is fixed
    assert out["obs"].shape == (256, 5, 64, 64) and out["info"].shape == (100, 40) and out["action"].shape == (100, 6)
    rows = [int(np.nonzero((sim.info.numpy() == r).all(1))[0][0]) for r in out["info"]]
    assert rows == sorted(set(rows))
    np.testing.assert_array_equal(out["reward"], sim.reward.numpy()[rows])
    np.testing.assert_array_equal(out["action"], action.numpy()[rows])
    # terminal observations: a sample of the 300 environments that finished in that step, with their indices
    fin = out["terminal_obs_env"].astype(np.int64)
    assert len(fin) == 256 and np.all(fin % 3 == 0) and np.all(np.diff(fin) > 0)
    np.testing.assert_array_equal(out["terminal_obs"], sim.terminal_obs.numpy()[fin])
    sim.done.zero_()
    bench.dump_outputs(str(tmp_path / "c"), sim, None)
    assert np.load(tmp_path / "c" / "terminal_obs.npy").shape == (0, 5, 64, 64) and not (tmp_path / "c" / "action.npy").exists()


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
