"""bench.py's reference arm (CPU only): one JSON line with the keys a caller of bench.py reads; on the GPU, the arrays
--dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600,
                       cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout


def _have_ref():
    return os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "stable_baselines3", "__init__.py"))


def test_reference_arm_line():
    """kind "reference" (the unmodified reference from baseline/_ref) when that copy exists, the oracle port otherwise."""
    out = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-steps", "12", "--ref-budget", "6"])
    lines = [l for l in out.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] and d["unit"] and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["config"]["workload"].startswith("HalfCheetah")
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if _have_ref() else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "K4" in cb["sample"]
    assert set(d["config"]) >= {"workload", "batch_size", "n_epochs", "rollouts", "n_steps", "parallelism"}
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    assert _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--cpu-steps", "12"], env).strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs holds the learner state after exactly warmup + steps iterations, taken before the e2e leg and the
    roofline touch the learner: bit-identical to a DeviceLearner run for 3 + 2 iterations (bench with the e2e leg) and for
    3 + 3 (bench without it).  float32 / float64 arrays, 64 MB at most.  That learner runs in a fresh interpreter, as bench
    does: the policy's orthogonal initialisation (a CPU QR) differs in the last bits with torch's thread count, which other
    tests in this process set."""
    def load(d):
        return {p.stem: np.load(p) for p in d.glob("*.npy")}

    script = ("import os, sys\nsys.path.insert(0, sys.argv[1])\nimport bench\n"
              "from icrl_b200.learner import WORKLOADS, DeviceLearner\n"
              "learner = DeviceLearner(WORKLOADS['halfcheetah'], seed=0, device='cuda', param_seed=0)\n"   # bench's rank 0
              "for it in range(1, 7):\n"
              "    learner.run()\n"
              "    if it >= 5:\n"
              "        bench.dump_outputs(learner, os.path.join(sys.argv[2], f'want{it}'))\n")
    r = subprocess.run([sys.executable, "-c", script, ROOT, str(tmp_path)], capture_output=True, text=True, timeout=600,
                       cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    want = {it: load(tmp_path / f"want{it}") for it in (5, 6)}
    quick = ["--warmup", "3", "--no-cpu", "--no-workloads", "--no-sweep"]
    for steps, extra in ((2, []), (3, ["--no-e2e"])):
        d = tmp_path / f"steps{steps}"
        lines = [l for l in _run(quick + ["--steps", str(steps), "--dump-outputs", str(d)] + extra).splitlines()
                 if l.startswith("{")]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
        got, ref = load(d), want[3 + steps]
        assert {"costs", "reward_advantages", "ppo_step_stats", "policy_params", "cn_params", "dual_state"} <= set(got)
        assert set(got) == set(ref) and sum(x.nbytes for x in got.values()) <= 64 * 1024 * 1024
        for k in got:
            assert got[k].dtype in (np.float32, np.float64), k
            np.testing.assert_array_equal(got[k], ref[k], err_msg=f"--steps {steps}: {k}")
    assert not np.array_equal(want[5]["policy_params"], want[6]["policy_params"])
