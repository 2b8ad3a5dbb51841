"""Whole-step time (CUDA graph, L2 flushed, mean over many steps) under different environment settings:
    python scripts/tune_step.py IMPALA_MLP_TC=0,1 [--config c4] [--steps 200]
One fresh engine (= fresh graph capture, the kernel choice is baked in at capture) per value."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from torched_impala_b200 import synth  # noqa: E402
from torched_impala_b200.engine import LearnerEngine  # noqa: E402
from torched_impala_b200.utils import default_hparams  # noqa: E402

CFG = {"c4": dict(T=20, B=4096, O=24, A=4, H=256), "c3": dict(T=20, B=1024, O=24, A=4, H=256),
       "c5": dict(T=100, B=8192, O=64, A=4, H=512)}
cfg, steps, sweeps = "c4", 200, []
args = sys.argv[1:]
while args:
    a = args.pop(0)
    if a == "--config":
        cfg = args.pop(0)
    elif a == "--steps":
        steps = int(args.pop(0))
    else:
        k, vals = a.split("=")
        sweeps.append((k, vals.split(",")))
w = CFG[cfg]
hp = default_hparams(batch_size=w["B"], max_timesteps=w["T"])
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
batch = synth.make_batch(1, w["T"], w["B"], w["O"], w["A"])
params = synth.init_params(0, w["O"], w["A"], w["H"])


def run(label):
    eng = LearnerEngine(w["T"], w["B"], w["O"], w["A"], w["H"], w["H"], hp)
    eng.load_state(params)
    eng.load_device_batch(batch)
    evs = []
    with torch.cuda.stream(eng.stream):
        for i in range(steps + 10):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(eng.stream)
            eng.step(0)
            e1.record(eng.stream)
            if i >= 10:
                evs.append((e0, e1))
    eng.synchronize()
    us = sum(a.elapsed_time(b) for a, b in evs) * 1e3 / len(evs)
    print(f"{label}: {us:.2f} us/step", flush=True)
    del eng


run("default")
for k, vals in sweeps:
    for v in vals:
        os.environ[k] = v
        run(f"{k}={v}")
    os.environ.pop(k)
