"""torchrun target: N-rank sharded learner steps vs a single-rank full-batch run.

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        tests/multi_gpu_check.py [--obs O] [--hidden H]

Every rank takes its B/N slice, all ranks all-reduce [gradient | loss scalars] once per step and
apply identical clip+Adam; rank 0 additionally replays the same batches on one GPU with the
full batch and compares loss scalars and parameters (float32 sum order differs -> ~1e-6).
The network shape picks the kernels: obs 24 / hidden 256 (default) runs the paired tensor-core
backward, which pushes the gradient itself; obs 64 / hidden 512 runs the wide kernels, followed by
the stand-alone push producer.
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from oracle.check import first_step_parity  # noqa: E402
from torched_impala_b200 import synth  # noqa: E402
from torched_impala_b200.engine import LearnerEngine  # noqa: E402
from torched_impala_b200.utils import default_hparams  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ap = argparse.ArgumentParser()
    ap.add_argument("--obs", type=int, default=24)
    ap.add_argument("--hidden", type=int, default=256)
    args = ap.parse_args()
    T, B, O, A, H = 20, 512, args.obs, 4, args.hidden
    hp = default_hparams(batch_size=B, max_timesteps=T)
    params = synth.init_params(3, O, A, H)
    batches = [synth.make_batch(10 + u, T, B, O, A, ragged=(u == 1)) for u in range(3)]
    eng = LearnerEngine(T, B // world, O, A, H, H, hp, global_batch=B, device=f"cuda:{local}",
                        process_group=dist.group.WORLD)
    # (1) against the float64 oracle of the FULL batch: every rank checks its shard's vs / pg_adv,
    # the oracle's scalar and gradient sums are all-reduced (oracle/check.py)
    par = first_step_parity(eng, params, synth.shard_batch(batches[0], rank, world), group=dist.group.WORLD)
    assert par["ok"], par
    # (2) against the single-GPU engine on the full batch, several updates
    eng.load_state(params)
    eng.adam_m.zero_(), eng.adam_v.zero_(), eng.adam_step.zero_()
    scal = []
    for u, b in enumerate(batches):
        eng.fill_host(synth.shard_batch(b, rank, world), u % 2)
        eng.ingest(u % 2)
        eng.step(u % 2)
        scal.append(eng.read_scalars())
    mine = eng.params.detach().clone()
    # replicas must stay bit-identical
    gathered = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(gathered, mine)
    for g in gathered:
        assert torch.equal(g, gathered[0]), "ranks diverged"
    if rank == 0:
        ref = LearnerEngine(T, B, O, A, H, H, hp, device=f"cuda:{local}")
        ref.load_state(params)
        for u, b in enumerate(batches):
            ref.fill_host(b, u % 2)
            ref.ingest(u % 2)
            ref.step(u % 2)
            want = ref.read_scalars()
            for k in ("value_fn_loss", "policy_loss", "policy_entropy", "total_loss", "batch_mean_reward"):
                assert abs(scal[u][k] - want[k]) < 1e-5 * max(1.0, abs(want[k])), (u, k, scal[u][k], want[k])
        d = (mine - ref.params).abs().max().item()
        assert d < 2e-5, d
        print(f"MULTI_GPU_OK world={world} allreduce={('peer(fused)' if eng.peer['fused'] else 'peer(standalone)') if eng.peer else 'nccl'} max|dparam|={d:.2e} "
              f"loss={scal[-1]['total_loss']:.6f} oracle: max|dvs|={par['max_abs_vs']:.1e} max|dscalar|={par['max_abs_scalar']:.1e} "
              f"rel|dgrad|={par['max_rel_grad']:.1e}")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
