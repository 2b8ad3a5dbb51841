"""CPU: the host side of the drop-in boundary - wire format, packing, C ABI, Learner surface."""
import os
import queue
import re

import numpy as np
import pytest
import torch

from conftest import PKEYS, ROOT
from oracle.cpu_learner_port import CpuLearnerPort
from oracle.impala_oracle import BatchedLearner
from torched_impala_b200 import _cabi, synth
from torched_impala_b200.learner import Learner, pack_trajectory
from torched_impala_b200.models import MlpPolicy, MlpValueFn
from torched_impala_b200.utils import Counter, Trajectory, default_hparams


def empty_views(T, B, O, A):
    return {"obs": np.full((T + 1, B, O), 7, np.float32), "beh_logits": np.full((T, B, A), 7, np.float32),
            "actions": np.full((T, B), 7, np.int32), "rewards": np.full((T, B), 7, np.float32),
            "done": np.full((T, B), 7, np.uint8), "lens": np.full((B,), 7, np.int32)}


@pytest.mark.parametrize("ragged", [False, True])
def test_pack_roundtrip(ragged):
    """Dense batch -> reference wire format -> pack_trajectory == the same dense batch."""
    T, B, O, A = 12, 9, 5, 3
    batch = synth.make_batch(3, T, B, O, A, ragged=ragged)
    views = empty_views(T, B, O, A)  # stale garbage everywhere: packing must overwrite/zero it
    total = 0.0
    for b, tr in enumerate(synth.to_trajectories(batch)):
        total += pack_trajectory(views, b, tr, T)
    for k in batch:
        np.testing.assert_array_equal(views[k], batch[k], err_msg=k)
    assert abs(total - batch["rewards"].astype(np.float64).sum()) < 1e-9


def test_pack_rejects_bad_trajectories():
    T, B, O, A = 6, 2, 3, 2
    trs = synth.to_trajectories(synth.make_batch(0, 8, B, O, A))
    with pytest.raises(ValueError):
        pack_trajectory(empty_views(T, B, O, A), 0, trs[0], T)  # longer than the unroll
    trs[1].obs.pop()
    with pytest.raises(ValueError):
        pack_trajectory(empty_views(8, B, O, A), 0, trs[1], 8)


def test_header_symbols_are_exported_and_bound():
    """Every function include/impala_b200.h declares is exported by the .so and has a ctypes
    signature (no compute call is made - there is no GPU here)."""
    hdr = open(os.path.join(ROOT, "include", "impala_b200.h")).read()
    declared = set(re.findall(r"^\s*(?:int64_t|long long|int)\s+(impala_\w+)\s*\(", hdr, flags=re.M))
    assert len(declared) >= 11
    assert declared == set(_cabi.SIGNATURES), declared ^ set(_cabi.SIGNATURES)
    lib = _cabi.lib()
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.impala_compiled_sm() == 100


def test_layouts():
    offs, total = _cabi.param_layout(24, 256, 4)
    assert offs == [0, 6144, 6400, 7424] and total == 7456 and all(o % 32 == 0 for o in offs)
    boffs, nbytes = _cabi.batch_layout(20, 4096, 24, 4)
    assert all(o % 256 == 0 for o in boffs) and nbytes % 256 == 0
    # algorithmic bytes of SURVEY.md 8d (c4) + one lens vector, modulo alignment padding
    algo = 4 * 21 * 4096 * 24 + 4 * 20 * 4096 * 4 + 4 * 20 * 4096 * 2 + 20 * 4096
    assert 0 <= nbytes - (algo + 4 * 4096) < 6 * 256
    assert _cabi.lib().impala_mlp_backward_workspace(1000, 200, 32, 2) == -2  # O > 64: loud, not silent


def test_learner_surface_and_no_cpu_fallback(tmp_path):
    """Constructor / attributes of reference learner.py:17-66,277-295; and on a machine without
    CUDA the update loop must raise, never fall back to a CPU path."""
    hp = default_hparams(batch_size=2, max_timesteps=5, max_updates=1, save_every=1)
    policy, value_fn = MlpPolicy(4, 2, 8), MlpValueFn(4, 8)
    policy.share_memory()
    lrn = Learner(1, hp, policy, value_fn, queue.Queue(), Counter(0), log_path=tmp_path / "logs")
    assert (tmp_path / "logs" / "l1").is_dir() and not lrn.completion.is_set()
    assert set(lrn.policy_weights) == set(PKEYS)
    assert all(v.dtype == torch.float64 for v in lrn.policy_weights.values())
    ck = tmp_path / "ck.pt"
    lrn.save(ck)
    blob = torch.load(ck)
    assert set(blob) == {"policy_state_dict", "value_fn_state_dict"}
    with torch.no_grad():
        policy.model[0].weight.zero_()
    lrn.load(ck)
    assert torch.equal(policy.state_dict()[PKEYS[0]], blob["policy_state_dict"][PKEYS[0]])
    if not torch.cuda.is_available():
        with pytest.raises(_cabi.ImpalaCudaError):
            lrn._learn()
        assert lrn.completion.is_set()


def test_unmodified_reference_actor_feeds_the_packer():
    """Trajectories the reference's own actor.py produced, run unmodified against the in-repo old-API
    CartPole (tests/golden/reference_actor/cartpole.npz, oracle/gen_golden.py), rebuilt in its wire
    format: (a) the packer accepts them and (b) they give the same update whether they go through
    the reference's per-trajectory path or through the packed dense batch."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "reference_actor", "cartpole.npz"))
    T, B = z["rewards"].shape
    hp = default_hparams(batch_size=B, max_timesteps=T, verbose=0)
    trajs = []
    for b, L in enumerate(z["lens"].tolist()):  # what actor.py appends per step: obs (O,) f64, a (1,) i64,
        tr = Trajectory((1, b + 1))             # r () f64, d () bool, logits (A,) f64
        tr.obs.append(torch.from_numpy(z["obs"][0, b]))
        for t in range(L):
            tr.add(torch.from_numpy(z["obs"][t + 1, b]), torch.from_numpy(z["actions"][t, b:b + 1]),
                   torch.tensor(z["rewards"][t, b]), torch.tensor(z["done"][t, b]), torch.from_numpy(z["logits"][t, b]))
        trajs.append(tr)
    assert all(1 <= len(t.r) <= T and len(t.obs) == len(t.r) + 1 for t in trajs)
    assert all(t.d[-1] or len(t.r) == T for t in trajs) and not any(d for t in trajs for d in t.d[:-1])
    views = empty_views(T, B, 4, 2)
    for b, tr in enumerate(trajs):
        pack_trajectory(views, b, tr, T)
    assert views["done"].sum() == sum(bool(t.d[-1]) for t in trajs)
    params = synth.init_params(5, 4, 2, 16)
    port = CpuLearnerPort(params, hp, threads=1).update(trajs)
    dense = BatchedLearner(params, hp).update(views)
    for k in ("value_fn_loss", "policy_loss", "policy_entropy", "total_loss", "batch_mean_reward"):
        # the packed batch is float32, the wire format float64: rounding of obs/logits only
        assert abs(port[k] - dense[k]) < 1e-5 * max(1.0, abs(port[k])), (k, port[k], dense[k])


def test_header_is_plain_c(tmp_path):
    """include/impala_b200.h is the drop-in boundary: it must compile as C99 (and as C++) on its own,
    and a C program must link against the shared library through it."""
    import shutil
    import subprocess

    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "use_abi.c"
    src.write_text('#include <stdio.h>\n#include "impala_b200.h"\n'
                   'int main(void) { int64_t off[4], total; int rc = impala_param_layout(24, 256, 4, off, &total);\n'
                   '  printf("%d %d %lld\\n", impala_abi_version(), rc, (long long)total); return rc; }\n')
    inc = os.path.join(ROOT, "include")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-fsyntax-only", "-I", inc, str(src)], check=True)
    subprocess.run(["g++", "-std=c++17", "-Wall", "-Werror", "-fsyntax-only", "-x", "c++", "-I", inc, str(src)], check=True)
    exe = tmp_path / "use_abi"
    libdir = os.path.dirname(_cabi.LIB_PATH)
    subprocess.run(["gcc", "-std=c99", "-I", inc, str(src), "-o", str(exe), "-L", libdir, "-limpala_b200",
                    f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert out[0] == "1" and out[1] == "0"
    assert int(out[2]) == _cabi.param_layout(24, 256, 4)[1]


def test_policy_snapshot_is_versioned():
    """SURVEY 8f-2: publications bump a shared version (odd while a write is in progress) and
    policy_snapshot() never returns a torn copy; policy_weights keeps the reference's semantics."""
    hp = default_hparams(batch_size=2, max_timesteps=5, max_updates=1)
    policy, value_fn = MlpPolicy(4, 2, 8), MlpValueFn(4, 8)
    policy.share_memory()
    lrn = Learner(1, hp, policy, value_fn, queue.Queue(), Counter(0))
    assert lrn.policy_version == 0
    v, sd = lrn.policy_snapshot()
    assert v == 0 and set(sd) == set(PKEYS)
    assert all(torch.equal(sd[k], policy.state_dict()[k]) and sd[k] is not policy.state_dict()[k] for k in PKEYS)
    lrn._version.value += 2  # what a completed publication does
    assert lrn.policy_version == 2 and lrn.policy_snapshot()[0] == 2


def test_shard_control_block_and_dp_config():
    """Host side of the data-parallel learner: control block shared by name, JSON-able config."""
    import json

    from torched_impala_b200 import dp

    ctl = dp.ShardControl()
    try:
        other = dp.ShardControl(ctl.name)
        ctl.w[dp._CMD] = 7
        ctl.w[dp._DMA_ACK + 3] = 5
        assert other.w[dp._CMD] == 7 and other.w[dp._DMA_ACK + 3] == 5 and other.w[dp._STOP] == 0
        other.close()
    finally:
        ctl.close()
    hp = default_hparams(batch_size=4, max_timesteps=5, log_path=None)
    lrn = Learner(2, hp, MlpPolicy(4, 2, 8), MlpValueFn(4, 8), queue.Queue(), Counter(0), devices=["cuda:0", "cuda:1"])
    cfg = lrn._cfg()
    assert json.loads(json.dumps(cfg))["B"] == 4 and cfg["H_pi"] == 8 and lrn.devices == ["cuda:0", "cuda:1"]
    with pytest.raises(ValueError):
        Learner(3, default_hparams(batch_size=3), MlpPolicy(4, 2, 8), MlpValueFn(4, 8), queue.Queue(), Counter(0),
                devices=["cuda:0", "cuda:1"])._make_engine(None, 2)
