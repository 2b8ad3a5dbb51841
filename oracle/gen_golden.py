"""TEST INFRASTRUCTURE - generate tests/golden/*.npz by running the REAL reference.

Run where the reference is importable ($IMPALA_REFERENCE_DIR, or oracle/_ref from oracle/make_ref.py):

    python -m oracle.gen_golden [name ...]      (default: every case, and the actor trajectories)

For every case below a seeded synthetic batch per update is converted to the
reference wire format (lists of float64 tensors), pushed through the unmodified
`/root/reference/learner.py::Learner._learn` via an in-process list queue, and the
numbers the reference exposes are recorded: the five TensorBoard scalars of every
update (`learner.py:217-240`) and both state_dicts after every update.  The
per-element tensors the reference keeps in locals (`vt`, `pg_adv`, `learner.py:127-135`)
and the raw gradients are taken from `oracle/cpu_learner_port.py`, after asserting
that the port reproduces the reference's scalars and parameters to 1e-12.  A case with
`sample=N` keeps every file under 1 MB: of each parameter larger than N entries, the parameters
after every update and the raw gradients are stored only at N seeded flat indices
(`sample_<net>_<key>`).

`reference_actor` records what the reference's own actor.py ships: it runs unmodified against
the in-repo old-API CartPole and its trajectories are stored densely (float64, zero padded).
"""
from __future__ import annotations

import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import refload  # noqa: E402
from oracle.cpu_learner_port import PKEYS, CpuLearnerPort  # noqa: E402
from torched_impala_b200 import synth  # noqa: E402
from torched_impala_b200.utils import default_hparams  # noqa: E402

CASES = {
    # name: dict(T, B, O, A, H_pi, H_v, ragged, unit_reward, updates, hp overrides)
    "c1_cartpole_ragged": dict(T=20, B=8, O=4, A=2, H_pi=32, H_v=32, ragged=True,
                               unit_reward=True, updates=3, hp={}),
    "c2_vtrace_fixed": dict(T=20, B=256, O=4, A=2, H_pi=32, H_v=32, ragged=False,
                            unit_reward=False, updates=2, hp={}),
    "c3_small_fixed": dict(T=20, B=64, O=24, A=4, H_pi=256, H_v=256, ragged=False,
                           unit_reward=False, updates=2, hp={}),
    "c3_small_ragged": dict(T=20, B=48, O=24, A=4, H_pi=256, H_v=256, ragged=True,
                            unit_reward=False, updates=2, hp={}),
    "c5_small_long": dict(T=100, B=16, O=64, A=4, H_pi=512, H_v=512, ragged=False,
                          unit_reward=False, updates=1, hp={}, sample=2048),
    "odd_shapes_clip": dict(T=12, B=32, O=7, A=3, H_pi=40, H_v=24, ragged=True,
                            unit_reward=False, updates=2,
                            hp=dict(max_norm=0.05, rho_bar=0.7, c_bar=0.9, entropy_c=0.01,
                                    v_loss_c=0.7, policy_loss_c=1.3, gamma=0.97, lr=3e-3)),
}


def run_reference(case, batches, params, hp):
    ref_learner, ref_models, ref_utils = refload.load()
    import torch

    torch.set_num_threads(1)
    ref_learner.SummaryWriter = refload.ScalarRecorder
    refload.ScalarRecorder.instances.clear()
    policy = ref_models.MlpPolicy(case["O"], case["A"], case["H_pi"])
    value_fn = ref_models.MlpValueFn(case["O"], case["H_v"])
    policy.load_state_dict({k: torch.tensor(v, dtype=torch.float64)
                            for k, v in params["policy"].items()})
    value_fn.load_state_dict({k: torch.tensor(v, dtype=torch.float64)
                              for k, v in params["value_fn"].items()})
    policy.eval()
    value_fn.eval()   # parity setting: Dropout(p=0.8) off (SURVEY.md section 0.4)
    trajs = []
    for b in batches:
        for tr in synth.to_trajectories(b):
            trajs.append(ref_utils.Trajectory(tr.id, tr.obs, tr.a, tr.r, tr.d, tr.logits))
    ref_hp = ref_utils.Hyperparameters(**hp._asdict())
    snaps = []

    def hook(step):
        snaps.append({"policy": {k: v.detach().numpy().copy() for k, v in policy.state_dict().items()},
                      "value_fn": {k: v.detach().numpy().copy() for k, v in value_fn.state_dict().items()}})

    refload.ScalarRecorder.hook = hook
    with tempfile.TemporaryDirectory() as tmp:
        lrn = ref_learner.Learner(1, ref_hp, policy, value_fn, refload.ListQueue(trajs),
                                  ref_utils.Counter(0), log_path=os.path.join(tmp, "log"))
        lrn._learn()
    refload.ScalarRecorder.hook = None
    rec = refload.ScalarRecorder.instances[-1].scalars
    per_update = [dict() for _ in batches]
    for tag, step, val in rec:
        per_update[step - 1][tag] = val
    return per_update, snaps


def reference_actor(out_dir, B=6, T=20, H=16):
    """B trajectories of the reference's actor.py (CartPole, policy hidden H, max_timesteps T)."""
    import queue

    import torch

    from oracle import cartpole_env

    refload.load(env_factory=cartpole_env.make)
    import actor as ref_actor
    import models as ref_models
    import utils as ref_utils

    hp = ref_utils.Hyperparameters(**default_hparams(batch_size=B, max_timesteps=T, verbose=0)._asdict())
    torch.manual_seed(0)
    shared = ref_models.MlpPolicy(4, 2, H)

    class FakeLearner:  # what actor.py touches: .completion.is_set() and .policy_weights
        class completion:
            calls = 0

            @classmethod
            def is_set(cls):
                cls.calls += 1
                return cls.calls > B

        policy_weights = shared.state_dict()

    q = queue.Queue()
    ref_actor.Actor(1, hp, ref_models.MlpPolicy(4, 2, H), FakeLearner, q, ref_utils.Counter(0))._act()
    trajs = [q.get_nowait() for _ in range(B)]
    blob = dict(meta_torch_version=np.array(torch.__version__), lens=np.zeros(B, np.int32),
                obs=np.zeros((T + 1, B, 4)), logits=np.zeros((T, B, 2)), actions=np.zeros((T, B), np.int64),
                rewards=np.zeros((T, B)), done=np.zeros((T, B), bool))
    for b, tr in enumerate(trajs):
        L = len(tr.r)
        blob["lens"][b] = L
        blob["obs"][:L + 1, b] = torch.stack(tr.obs).numpy()
        blob["logits"][:L, b] = torch.stack(tr.logits).detach().numpy()
        blob["actions"][:L, b] = torch.cat(tr.a).numpy()
        blob["rewards"][:L, b] = torch.stack(tr.r).numpy()
        blob["done"][:L, b] = torch.stack(tr.d).numpy()
    os.makedirs(os.path.join(out_dir, "reference_actor"), exist_ok=True)
    path = os.path.join(out_dir, "reference_actor", "cartpole.npz")
    np.savez_compressed(path, **blob)
    print(f"reference_actor: lens {blob['lens'].tolist()} -> {path} ({os.path.getsize(path) / 1024:.0f} KiB)")


def main(names):
    import torch

    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    if not names or "reference_actor" in names:
        reference_actor(out_dir)
    for name, case in CASES.items():
        if names and name not in names:
            continue
        seed = sum(map(ord, name)) % 1000
        hp = default_hparams(batch_size=case["B"], max_updates=case["updates"],
                             max_timesteps=case["T"], policy_hidden_dims=case["H_pi"],
                             value_fn_hidden_dims=case["H_v"], save_every=10 ** 9,
                             eval_every=None, verbose=0, **case["hp"])
        params = synth.init_params(seed, case["O"], case["A"], case["H_pi"], case["H_v"])
        batches = [synth.make_batch(seed + 1 + u, case["T"], case["B"], case["O"], case["A"],
                                    ragged=case["ragged"], unit_reward=case["unit_reward"])
                   for u in range(case["updates"])]
        ref_scalars, ref_snaps = run_reference(case, batches, params, hp)

        port = CpuLearnerPort(params, hp, threads=1)
        blob = {"meta_torch_version": np.array(torch.__version__),
                "meta_case": np.array(repr(case)), "meta_hp": np.array(repr(hp._asdict()))}
        for k, v in hp._asdict().items():
            if isinstance(v, (int, float)) and not isinstance(v, bool):
                blob[f"hp_{k}"] = np.array(v)
        keep = {}  # (net, key) -> flat indices stored of the parameters after each update and the raw gradients
        for grp in ("policy", "value_fn"):
            for k in PKEYS:
                blob[f"init_{grp}_{k}"] = params[grp][k]
                n = params[grp][k].size
                if case.get("sample") and n > case["sample"]:
                    idx = np.sort(np.random.default_rng(seed).choice(n, case["sample"], replace=False))
                    keep[grp, k] = blob[f"sample_{grp}_{k}"] = idx.astype(np.int32)

        def stored(grp, k, arr):
            return arr.reshape(-1)[keep[grp, k]] if (grp, k) in keep else arr

        worst = 0.0
        for u, batch in enumerate(batches):
            res = port.update(synth.to_trajectories(batch), keep_elements=True)
            for tag in ("value_fn_loss", "policy_loss", "policy_entropy", "total_loss",
                        "batch_mean_reward"):
                d = abs(res[tag] - ref_scalars[u][tag])
                worst = max(worst, d)
                assert d <= 1e-12 * max(1.0, abs(ref_scalars[u][tag])), (name, u, tag, d)
                blob[f"u{u}_{tag}"] = np.array(ref_scalars[u][tag])
            st = port.state()
            for grp in ("policy", "value_fn"):
                for k in PKEYS:
                    d = np.abs(st[grp][k] - ref_snaps[u][grp][k]).max()
                    worst = max(worst, float(d))
                    assert d <= 1e-12, (name, u, grp, k, d)
                    blob[f"u{u}_{grp}_{k}"] = stored(grp, k, ref_snaps[u][grp][k])
            T, B = case["T"], case["B"]
            vs = np.zeros((T + 1, B))
            pg = np.zeros((T, B))
            for b, (tgt, adv) in enumerate(res["elements"]):
                L = adv.shape[0]
                vs[:L + 1, b] = tgt.numpy()
                pg[:L, b] = adv.numpy()
            blob[f"u{u}_vs"] = vs
            blob[f"u{u}_pg_adv"] = pg
            for i, (grp, k) in enumerate([(g, k) for g in ("policy", "value_fn") for k in PKEYS]):
                blob[f"u{u}_rawgrad_{grp}_{k}"] = stored(grp, k, res["raw_grads"][i].numpy())
            for k, v in batch.items():
                blob[f"u{u}_in_{k}"] = v
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **blob)
        print(f"{name}: port-vs-reference worst abs diff {worst:.3e} -> {path} "
              f"({os.path.getsize(path) / 1024:.0f} KiB)")


if __name__ == "__main__":
    main(sys.argv[1:])
