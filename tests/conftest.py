"""pytest wiring: the `gpu` marker, repo-root imports and golden-fixture loading."""
import ast
import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
PKEYS = ("model.0.weight", "model.0.bias", "model.3.weight", "model.3.bias")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def golden_names():
    return sorted(os.path.splitext(os.path.basename(p))[0]
                  for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


class Golden:
    """One tests/golden/*.npz produced by oracle/gen_golden.py from the real reference."""

    def __init__(self, name):
        from torched_impala_b200.utils import default_hparams

        self.name = name
        self.z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        self.case = ast.literal_eval(str(self.z["meta_case"]))
        hp = ast.literal_eval(str(self.z["meta_hp"]))
        self.hp = default_hparams(**hp)
        self.updates = self.case["updates"]

    def init_params(self):
        return {g: {k: self.z[f"init_{g}_{k}"] for k in PKEYS} for g in ("policy", "value_fn")}

    def batch(self, u):
        return {k: self.z[f"u{u}_in_{k}"] for k in
                ("obs", "beh_logits", "actions", "rewards", "done", "lens")}

    def scalars(self, u):
        return {k: float(self.z[f"u{u}_{k}"]) for k in
                ("value_fn_loss", "policy_loss", "policy_entropy", "total_loss",
                 "batch_mean_reward")}

    def params_after(self, u):
        return {g: {k: self.z[f"u{u}_{g}_{k}"] for k in PKEYS} for g in ("policy", "value_fn")}

    def raw_grads(self, u):
        return {g: {k: self.z[f"u{u}_rawgrad_{g}_{k}"] for k in PKEYS}
                for g in ("policy", "value_fn")}

    def pick(self, g, k, arr):
        """`arr`, a full parameter-shaped array, at the entries params_after / raw_grads hold for it:
        the files of the large networks keep those at a seeded sample of flat indices only."""
        name = f"sample_{g}_{k}"
        return np.asarray(arr).reshape(-1)[self.z[name]] if name in self.z.files else arr


@pytest.fixture(params=golden_names())
def golden(request):
    return Golden(request.param)
