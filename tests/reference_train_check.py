"""Run the reference's OWN `train.py` + `actor.py` (unmodified, from oracle/_ref) against the B200 Learner.

BASELINE.json configs[0] (c1): CartPole, 2 CPU actors, T=20, batch=8, hidden=32.  Executed by
test_gpu_reference_train.py in a fresh interpreter.  Nothing of the reference is edited:

  * `from learner import Learner` (train.py:7, actor.py:10) resolves to `torched_impala_b200.learner`
    - the one-line swap of INTEGRATION.md section 1, done here through `sys.modules`;
  * train.py hard-codes its hyper-parameters (train.py:11-36, README TODO "Add command line argument
    support"): `utils.Hyperparameters` is wrapped so the literal call yields the c1 values;
  * the GPUs are hidden from the launcher and the actors (the reference picks its device at import:
    models.py:5, actor.py:13), the learner process gets them back (IMPALA_LEARNER_VISIBLE_DEVICES);
  * `gym.make` is the in-repo old-API CartPole (oracle/_ref/gym stub).
Checks afterwards: exit through the reference's own shutdown path, every update counted, the
checkpoint of train.py's `save_every` written and loadable by the reference's test.py code path,
TensorBoard files of learner and both actors present, the shared policy changed.
"""
import os
import runpy
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")


def main():
    out_dir = sys.argv[1]
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    os.environ["IMPALA_LEARNER_VISIBLE_DEVICES"] = vis if vis not in (None, "") else "0"
    os.environ["CUDA_VISIBLE_DEVICES"] = ""           # launcher + actors stay on the CPU
    os.environ["PYTORCH_NVML_BASED_CUDA_CHECK"] = "1"  # torch.cuda.is_available() without cuInit in the parent
    sys.path.insert(0, ROOT)
    sys.path.insert(0, REF)
    if not os.path.isfile(os.path.join(REF, "train.py")):
        print("oracle/_ref missing: run python -m oracle.make_ref (copies it from the reference checkout)")
        sys.exit(2)
    import torch

    assert not torch.cuda.is_available()
    import utils as ref_utils  # oracle/_ref/utils.py (imports the gym stub)

    import torched_impala_b200.learner as b200_learner

    sys.modules["learner"] = b200_learner               # train.py:7 / actor.py:10
    real_hp = ref_utils.Hyperparameters
    c1 = dict(max_updates=6, policy_hidden_dims=32, value_fn_hidden_dims=32, batch_size=8, max_timesteps=20,
              n_actors=2, log_path=out_dir, save_every=3, eval_every=2, eval_eps=3, verbose=1)

    def hp_c1(**kw):
        kw.update(c1)
        return real_hp(**kw)

    ref_utils.Hyperparameters = hp_c1
    os.chdir(out_dir)
    runpy.run_path(os.path.join(REF, "train.py"), run_name="__main__")   # returns after terminate/join
    # ---- post-mortem
    runs = [d for d in os.listdir(out_dir) if os.path.isdir(os.path.join(out_dir, d))]
    assert len(runs) == 1, runs
    run = os.path.join(out_dir, runs[0])
    assert os.path.isfile(os.path.join(run, "hyperparameters.txt"))
    for sub in ("l1", "a1", "a2"):
        files = os.listdir(os.path.join(run, sub))
        assert any(f.startswith("events.out.tfevents") for f in files), (sub, files)
    cks = sorted(f for f in os.listdir(os.path.join(run, "l1")) if f.endswith(".pt"))
    assert cks == ["IMPALA_CartPole-v1_l1_3.pt", "IMPALA_CartPole-v1_l1_6.pt"], cks
    import models as ref_models

    blob = torch.load(os.path.join(run, "l1", cks[-1]))
    pol = ref_models.MlpPolicy(4, 2, 32)                 # what reference test.py:62-65 does
    pol.load_state_dict(blob["policy_state_dict"])
    fresh = ref_models.MlpPolicy(4, 2, 32).state_dict()
    assert any(not torch.equal(fresh[k], v) for k, v in pol.state_dict().items())
    assert all(v.dtype == torch.float64 for v in blob["value_fn_state_dict"].values())
    print(f"REFERENCE_TRAIN_OK checkpoints={cks}")


if __name__ == "__main__":
    main()
