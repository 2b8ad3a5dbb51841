"""GPU: the reference's unmodified train.py + actor.py (oracle/_ref) drive the B200 Learner - c1.

BASELINE.json configs[0]: CartPole-v1, 2 CPU actors, T=20, batch=8, hidden=32.  See
tests/reference_train_check.py for what is (not) touched."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_unmodified_train_py_runs_against_the_b200_learner(tmp_path):
    if not os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "train.py")):
        pytest.fail("oracle/_ref is missing: __graft_entry__.build() / python -m oracle.make_ref creates it "
                    "from the reference checkout (oracle/make_ref.py)")
    script = os.path.join(os.path.dirname(__file__), "reference_train_check.py")
    out = tmp_path / "logs"
    out.mkdir()
    res = subprocess.run([sys.executable, script, str(out)], capture_output=True, text=True, timeout=600)
    tail = res.stdout[-4000:] + res.stderr[-4000:]
    assert res.returncode == 0, tail
    assert "REFERENCE_TRAIN_OK" in res.stdout, tail
    assert "[learner_1] update 6" in res.stdout and "evaluation reward" in res.stdout, tail
    assert "[actor_1] Finished acting" in res.stdout and "[actor_2] Finished acting" in res.stdout, tail
