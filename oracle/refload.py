"""TEST INFRASTRUCTURE - import the unmodified reference modules in this container.

`/root/reference/utils.py:6-7` imports `gym` and `pybullet_envs`, neither of which is
installed; two empty stub modules make `learner`, `models`, `utils`, `actor` import
cleanly (SURVEY.md section 8c).  `device` is resolved at import time
(`learner.py:13`), so CUDA is hidden first.  On the GPU box `/root/reference`
does not exist; the modules then come from `oracle/_ref/` (see oracle/make_ref.py).
"""
from __future__ import annotations

import os
import sys
import types

_HERE = os.path.dirname(os.path.abspath(__file__))


def reference_dir():
    """Where the unmodified reference modules can be imported from: $IMPALA_REFERENCE_DIR, or the
    copy oracle/make_ref.py left under the git-ignored oracle/_ref/."""
    for d in (os.environ.get("IMPALA_REFERENCE_DIR"), os.path.join(_HERE, "_ref")):
        if d and os.path.isfile(os.path.join(d, "learner.py")):
            return d
    return None


def available() -> bool:
    return reference_dir() is not None


def load(env_factory=None):
    """Returns the reference's (learner, models, utils) modules.

    env_factory, if given, becomes `gym.make` (used to run the unmodified actor.py
    against an in-repo old-API environment).
    """
    ref_dir = reference_dir()
    if ref_dir is None:
        raise RuntimeError("reference not found (set IMPALA_REFERENCE_DIR or run python -m oracle.make_ref)")
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    if "torch" in sys.modules:
        import torch

        if torch.cuda.is_available():  # `device` is resolved at import (learner.py:13, models.py:5)
            raise RuntimeError("import the reference in a process that has not initialised CUDA "
                               "(CUDA_VISIBLE_DEVICES must be empty before torch is imported)")
    if "gym" not in sys.modules:
        gym = types.ModuleType("gym")
        gym.Env = object
        sys.modules["gym"] = gym
    if env_factory is not None:
        sys.modules["gym"].make = env_factory
    sys.modules.setdefault("pybullet_envs", types.ModuleType("pybullet_envs"))
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import learner as ref_learner  # noqa: E402
    import models as ref_models  # noqa: E402
    import utils as ref_utils  # noqa: E402

    return ref_learner, ref_models, ref_utils


class ListQueue:
    """Duck-typed stand-in for mp.Queue: `get(timeout=)` pops from a python list."""

    def __init__(self, items):
        self.items = list(items)
        self.pos = 0

    def get(self, timeout=None):
        import queue

        if self.pos >= len(self.items):
            raise queue.Empty
        it = self.items[self.pos]
        self.pos += 1
        return it


class ScalarRecorder:
    """Replaces `learner.SummaryWriter`; records every add_scalar call."""

    instances = []
    hook = None  # called as hook(step) right after each update's total_loss is logged

    def __init__(self, *a, **k):
        self.scalars = []
        ScalarRecorder.instances.append(self)

    def add_text(self, *a, **k):
        pass

    def add_scalar(self, tag, value, step):
        try:
            value = float(value)
        except TypeError:
            value = float(value.item())
        self.scalars.append((tag.split("/")[-1], step, value))
        if tag.endswith("total_loss") and ScalarRecorder.hook is not None:
            ScalarRecorder.hook(step)

    def close(self):
        pass
