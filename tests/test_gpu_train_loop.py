"""GPU: a training run with forked CPU actor processes drives the B200 Learner - c1.

BASELINE.json configs[0]: CartPole-v1, 2 CPU actors, T=20, batch=8, hidden=32.  See
tests/train_loop_check.py for what the launcher does."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu


def test_train_loop_with_actor_processes_runs_against_the_b200_learner(tmp_path):
    script = os.path.join(os.path.dirname(__file__), "train_loop_check.py")
    out = tmp_path / "logs"
    out.mkdir()
    res = subprocess.run([sys.executable, script, str(out)], capture_output=True, text=True, timeout=600)
    tail = res.stdout[-4000:] + res.stderr[-4000:]
    assert res.returncode == 0, tail
    assert "TRAIN_LOOP_OK" in res.stdout, tail
    assert "[learner_1] update 6" in res.stdout and "evaluation reward" in res.stdout, tail
    assert "[actor_1] Finished acting" in res.stdout and "[actor_2] Finished acting" in res.stdout, tail
