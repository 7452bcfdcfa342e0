"""CPU: the reference arm of bench.py (`--impl reference`: the UNMODIFIED reference's CPU learner from oracle/_ref) prints exactly
one JSON line on stdout with the keys that readers of the bench line use, whatever libraries print meanwhile.

build() installs the reference under oracle/_ref only where the reference checkout is readable.  Elsewhere the arm runs with
the oracle's restatement of the same CPU learner (oracle/cpu_learner.py, pinned to the reference by tests/test_oracle.py)
in its place, and that learner prints to stdout on every step, so the output contract is checked on every machine."""
import json
import os
import subprocess
import sys

from oracle import ref_shim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# bench.py with the reference learner replaced by the oracle's CPU learner on the same recipe rollout
_STAND_IN = """
import os
import sys
sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import bench
from helpers import POLICY_CFG, load_golden, recipe_state_dict
from oracle.cpu_learner import CpuLearner


def make_cpu_learner(T=bench.CPU_SAMPLE["T"], N=bench.CPU_SAMPLE["N"]):
    learner = CpuLearner(recipe_state_dict(load_golden("full256")["shapes"], 5), POLICY_CFG)
    bufs, next_value = bench._recipe_rollout(T, N)

    def step():
        print("stand-in learner step")
        return learner.update(dict(bufs), next_value, T)
    return step, T * N


bench._make_cpu_learner = make_cpu_learner
sys.argv[0] = "bench.py"
bench.main()
"""


def _reference_arm():
    if ref_shim.reference_available():
        return [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"]
    return [sys.executable, "-c", _STAND_IN, "--impl", "reference"]


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="8", HB200_CPU_SAMPLE="16,4")
    p = subprocess.run(_reference_arm() + ["--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("DD-PPO learner frames/sec")
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"] > 0
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert p.returncode == 0 and p.stdout.strip() == ""
