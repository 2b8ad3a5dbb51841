"""A whole IMPALA training run - CPU actor processes, a bounded mp.Queue, fork - on the B200 Learner.

BASELINE.json configs[0] (c1): CartPole, 2 CPU actors, T=20, batch=8, hidden=32.  Executed by
test_gpu_train_loop.py in a fresh interpreter.  The launcher drives the Learner only through the
surface a training script uses (INTEGRATION.md section 1):

  * `Learner(id, hparams, policy, value_fn, q, update_counter, log_path)`, `start()`, `completion`,
    `terminate()`, `join()`; the actors read `learner.completion` and `learner.policy_weights`;
  * the GPUs are hidden from the launcher and the actors (CPU float64 policies, fork start method),
    the learner process gets them back (IMPALA_LEARNER_VISIBLE_DEVICES);
  * the environment is the in-repo old-API CartPole, evaluation a greedy rollout of it.
Checks afterwards: every update counted, the checkpoints of `save_every` written and loadable into a
fresh policy, the learner's TensorBoard file present, the shared policy changed.
"""
import os
import queue
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C1 = dict(max_updates=6, policy_hidden_dims=32, value_fn_hidden_dims=32, batch_size=8, max_timesteps=20,
          n_actors=2, save_every=3, eval_every=2, eval_eps=3, verbose=1)


def evaluate(policy, hp):
    """Mean and spread of the greedy episode return over hp.eval_eps CartPole episodes."""
    import torch

    from oracle.cartpole_env import make

    env, rewards = make(hp.env_name, seed=1000), []
    with torch.no_grad():
        for _ in range(hp.eval_eps):
            obs, total = env.reset(), 0.0
            for _ in range(hp.max_timesteps):
                a, _ = policy.select_action(torch.tensor(obs, dtype=torch.float64), deterministic=True)
                obs, r, d, _ = env.step(a.item())
                total += r
                if d:
                    break
            rewards.append(total)
    return float(np.mean(rewards)), float(np.std(rewards))


def act(actor_id, hp, policy, learner, q, done):
    """One actor process: roll CartPole episodes (at most max_timesteps steps) with the latest
    published weights and ship them in the reference wire format until the learner completes."""
    import torch

    from oracle.cartpole_env import make
    from torched_impala_b200.utils import Trajectory

    for p in policy.parameters():
        p.requires_grad = False
    env, n = make(hp.env_name, seed=actor_id), 0
    while not learner.completion.is_set():
        n += 1
        policy.load_state_dict(learner.policy_weights)
        obs = torch.tensor(env.reset(), dtype=torch.float64)
        traj = Trajectory((actor_id, n))
        traj.obs.append(obs)
        for _ in range(hp.max_timesteps):
            a, logits = policy.select_action(obs)
            o, r, d, _ = env.step(a.item())
            obs = torch.tensor(o, dtype=torch.float64)
            traj.add(obs, a, torch.tensor(r, dtype=torch.float64), torch.tensor(d), logits)
            if d:
                break
        while True:
            try:
                q.put(traj, timeout=1)
                break
            except queue.Full:
                if learner.completion.is_set():
                    break
    print(f"[actor_{actor_id}] Finished acting", flush=True)
    done.set()


def main():
    out_dir = sys.argv[1]
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    os.environ["IMPALA_LEARNER_VISIBLE_DEVICES"] = vis if vis not in (None, "") else "0"
    os.environ["CUDA_VISIBLE_DEVICES"] = ""           # launcher + actors stay on the CPU
    os.environ["PYTORCH_NVML_BASED_CUDA_CHECK"] = "1"  # torch.cuda.is_available() without cuInit in the parent
    sys.path.insert(0, ROOT)
    import torch
    import torch.multiprocessing as mp

    from torched_impala_b200.learner import Learner
    from torched_impala_b200.models import MlpPolicy, MlpValueFn
    from torched_impala_b200.utils import Counter, default_hparams

    assert not torch.cuda.is_available()
    mp.set_start_method("fork", force=True)
    run = os.path.join(out_dir, "run")
    hp = default_hparams(log_path=run, **C1)
    torch.manual_seed(0)
    q = mp.Queue(maxsize=hp.queue_lim)
    counter = Counter(0)
    policy = MlpPolicy(4, 2, hp.policy_hidden_dims)
    policy.share_memory()
    init = {k: v.clone() for k, v in policy.state_dict().items()}
    learner = Learner(1, hp, policy, MlpValueFn(4, hp.value_fn_hidden_dims), q, counter, run,
                      evaluator=lambda pol: evaluate(pol, hp))
    actors = []
    for i in range(1, hp.n_actors + 1):
        done = mp.Event()
        actors.append((mp.Process(target=act, args=(i, hp, MlpPolicy(4, 2, hp.policy_hidden_dims), learner, q, done),
                                  name=f"actor_{i}"), done))
    for p, _ in actors:
        p.start()
    learner.start()
    assert learner.completion.wait(timeout=300), "learner never signalled completion"
    for _, done in actors:
        assert done.wait(timeout=60), "an actor did not finish"
    learner.terminate()
    for p, _ in actors:
        p.terminate()
    learner.join()
    for p, _ in actors:
        p.join()
    # ---- post-mortem
    assert counter.value == hp.max_updates, counter.value
    files = os.listdir(os.path.join(run, "l1"))
    assert any(f.startswith("events.out.tfevents") for f in files), files
    cks = sorted(f for f in files if f.endswith(".pt"))
    assert cks == ["IMPALA_CartPole-v1_l1_3.pt", "IMPALA_CartPole-v1_l1_6.pt"], cks
    blob = torch.load(os.path.join(run, "l1", cks[-1]))
    pol = MlpPolicy(4, 2, hp.policy_hidden_dims)
    pol.load_state_dict(blob["policy_state_dict"])
    assert any(not torch.equal(init[k], v) for k, v in pol.state_dict().items())
    assert any(not torch.equal(init[k], v) for k, v in policy.state_dict().items())  # seen through shared memory
    assert all(v.dtype == torch.float64 for v in blob["value_fn_state_dict"].values())
    print(f"TRAIN_LOOP_OK checkpoints={cks}")


if __name__ == "__main__":
    main()
