"""bench.py's command line: the reference arm's JSON line and the argument checks on the CPU, the outputs
--dump-outputs writes on a GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, MPCB_CPU_SAMPLE_SECONDS="0.5")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "rollouts/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["config"]["workload"].startswith("cfg2")


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "error" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_steps_answers(tmp_path):
    """--dump-outputs writes cost / index / traj / first_control of every robot of the last timed step, in float64,
    and they are the float64 C oracle's answers for the seeded scenarios."""
    import numpy as np

    from oracle import c_oracle as K
    from oracle import closed_form as C

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--no-legs", "--no-cpu",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    out = {k: np.load(tmp_path / (k + ".npy")) for k in ("cost", "index", "traj", "first_control")}
    n = 1024
    assert {k: a.shape for k, a in out.items()} == dict(cost=(n,), index=(n,), traj=(n, 3, 3), first_control=(n, 2))
    assert all(a.dtype == np.float64 for a in out.values())
    V, B = C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0)
    scen = C.random_scenarios(n, 0)
    for i in (0, n - 1):
        o = K.solve_full(scen[i, :3], scen[i, 3:5], scen[i, :2], V, B, 3, C.COST_MM)
        assert out["index"][i] == o["index"] and abs(out["cost"][i] - o["cost"]) <= 1e-12 * o["cost"]
        np.testing.assert_allclose(out["traj"][i], o["traj"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(out["first_control"][i], o["first_control"], rtol=0, atol=1e-12)
