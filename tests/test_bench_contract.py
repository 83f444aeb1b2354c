"""bench.py's command line.  Without a GPU, the reference arm: ONE JSON line on stdout with the keys its readers use,
whatever libraries print while it runs.  On a GPU, the b200 arm: --steps timed steps and the --dump-outputs files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["value"] > 0 and d["gpu_launches"] == 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # exactly K timed steps: ms_per_step is the measured wall time of a step (nothing extrapolated)
    per_step = int(d["step_definition"].split("(")[1].split()[0])
    assert abs(d["value"] - per_step * d["steps"] / (d["ms_per_step"] * d["steps"] * 1e-3)) < 1e-6 * d["value"]


def test_reference_arm_other_ranks_stay_silent():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_steps_below_one_are_refused():
    for impl in ("reference", "b200"):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", impl, "--steps", "0"],
                           capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert p.returncode == 2 and p.stdout.strip() == "" and "--steps" in p.stderr


@pytest.mark.gpu
def test_b200_arm_times_k_steps_and_dumps_the_last(cuda, tmp_path):
    """K timed steps are K launches of the env step, and --dump-outputs holds what the last of them returned: the same
    seeded envs and action bank, replayed here, give the dumped arrays bit for bit in the last timed step only."""
    import torch
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    K = 3
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(K), "--warmup", "1", "--skip-cpu",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout[:500]
    d = json.loads(lines[0])
    assert d["steps"] == K and d["gpu_launches"] == K
    out = {f[:-len(".npy")]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype == np.float32 for a in out.values()) and sum(a.nbytes for a in out.values()) <= 64 << 20
    # the bench's inputs: seeded envs, a seeded action bank, pre-roll, W warm-up steps, then the K timed steps
    c, W = d["config"], d["warmup"]
    E = c["envs_per_gpu"]
    venv = BlueSkyVectorEnv("HorizontalCREnv-v0", E, device=0, seed=0, cd_enabled=True, n_intruders=c["n_intruders"],
                            autoreset_mode="same_step")
    venv.reset_torch()
    g = torch.Generator(device=cuda).manual_seed(1234)
    bank = torch.rand((K + W, E, 1), generator=g, device=cuda) * 2.0 - 1.0
    for i in range(c["preroll_steps"]):
        venv.step_torch(bank[i % (K + W)])
    for i in range(W):
        venv.step_torch(bank[i])
    for i in range(K):
        obs, rew, term, trunc = venv.step_torch(bank[W + i])
        want = {"obs_" + k: v for k, v in obs.items()}
        want.update(reward=rew, terminated=term, truncated=trunc)
        want = {k: v.float().cpu().numpy() for k, v in want.items()}
        assert set(out) == set(want)
        same = all(np.array_equal(out[k], want[k]) for k in want)
        assert same == (i == K - 1), f"timed step {i}: dump {'equals' if same else 'differs from'} the replay"
    venv.close()
