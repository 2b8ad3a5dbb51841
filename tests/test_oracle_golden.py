"""CPU: both oracle restatements against the golden vectors of the real reference.

The fixtures were produced by running the unmodified reference learner.py
(oracle/gen_golden.py); these tests pin the oracle without needing the reference.
"""
import numpy as np
import pytest

from conftest import PKEYS
from oracle.cpu_learner_port import CpuLearnerPort
from oracle.impala_oracle import BatchedLearner
from torched_impala_b200 import synth

SCALARS = ("value_fn_loss", "policy_loss", "policy_entropy", "total_loss", "batch_mean_reward")


def test_batched_oracle_matches_reference(golden):
    lrn = BatchedLearner(golden.init_params(), golden.hp)
    for u in range(golden.updates):
        out = lrn.update(golden.batch(u))
        ref = golden.scalars(u)
        for k in SCALARS:
            assert abs(out[k] - ref[k]) <= 1e-11 * max(1.0, abs(ref[k])), (k, out[k], ref[k])
        np.testing.assert_allclose(out["vs"], golden.z[f"u{u}_vs"], rtol=0, atol=1e-11)
        np.testing.assert_allclose(out["pg_adv"], golden.z[f"u{u}_pg_adv"], rtol=0, atol=1e-11)
        rg = golden.raw_grads(u)
        for g, got in (("policy", out["g_policy"]), ("value_fn", out["g_value"])):
            for k, arr in zip(PKEYS, got):
                np.testing.assert_allclose(golden.pick(g, k, arr), rg[g][k], rtol=0, atol=1e-11)
        st, want = lrn.state(), golden.params_after(u)
        for g in st:
            for k in PKEYS:
                np.testing.assert_allclose(golden.pick(g, k, st[g][k]), want[g][k], rtol=0, atol=1e-11)


def test_per_trajectory_port_matches_reference(golden):
    port = CpuLearnerPort(golden.init_params(), golden.hp, threads=1)
    for u in range(golden.updates):
        res = port.update(synth.to_trajectories(golden.batch(u)))
        ref = golden.scalars(u)
        for k in SCALARS:
            assert abs(res[k] - ref[k]) <= 1e-12 * max(1.0, abs(ref[k]))
        st, want = port.state(), golden.params_after(u)
        for g in st:
            for k in PKEYS:
                np.testing.assert_allclose(golden.pick(g, k, st[g][k]), want[g][k], rtol=0, atol=1e-12)


def test_reference_quirks_are_not_silently_fixed(golden):
    """mode="paper" (v[:-1], no second v[i+1] subtraction) must NOT match learner.py."""
    lrn = BatchedLearner(golden.init_params(), golden.hp)
    out = lrn.forward_backward(golden.batch(0), mode="paper")
    assert np.abs(out["vs"] - golden.z["u0_vs"]).max() > 1e-3


def test_padding_is_neutral():
    """A ragged batch equals the same trajectories padded into a longer unroll."""
    from torched_impala_b200.utils import default_hparams

    hp = default_hparams(batch_size=6)
    params = synth.init_params(3, 5, 3, 16)
    b = synth.make_batch(11, 9, 6, 5, 3, ragged=True)
    wide = {}
    for k, v in b.items():
        if k == "lens":
            wide[k] = v
        else:
            pad = np.zeros((4,) + v.shape[1:], v.dtype)
            wide[k] = np.concatenate([v, pad], 0)
    a = BatchedLearner(params, hp).forward_backward(b)
    w = BatchedLearner(params, hp).forward_backward(wide)
    for k in SCALARS[:4]:
        assert abs(a[k] - w[k]) < 1e-13
    for ga, gw in zip(a["g_policy"] + a["g_value"], w["g_policy"] + w["g_value"]):
        np.testing.assert_allclose(ga, gw, rtol=0, atol=1e-13)
