#!/usr/bin/env python
"""Learner steps/sec on synthetic (T=20, B=4096, O=24, A=4, H=256) trajectories.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Own arm (default): one process per GPU (torchrun for N > 1), global batch B=4096 sharded
B/N per rank ("scaling": "strong"), one all-reduce of [gradient | loss scalars] per step (done by the
optimizer kernel over NVLink peer memory; NCCL with IMPALA_ALLREDUCE=nccl).
  value  : learner steps/s with the batch already resident in HBM; each of the K timed steps
           is bracketed by CUDA events on the launching stream, L2 flushed between steps
  e2e    : the same through the host-facing API - every step copies that step's inputs from
           pinned host memory (one DMA), runs the update and reads the loss scalars back
  roofline / kernels : per-kernel CUDA-event timings of the same launch sequence (eager, L2
           flushed) against the binding roof of each kernel (HBM for V-trace/loss/optimizer,
           FP32 FMA pipe for the MLP kernels - see DESIGN.md)
  cpu_baseline : the per-trajectory float64 torch port of learner.py (oracle/) on host cores
Reference arm (--impl reference): rank 0 times that CPU port alone and prints its own line.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs[2..4]; c4 is the configuration the metric is quoted on (the default).
WORKLOADS = {
    "c3": dict(T=20, B=1024, O=24, A=4, H=256,
               name="c3: synthetic obs=24 act=4 hidden=256, T=20 B=1024 (BASELINE.json configs[2])"),
    "c4": dict(T=20, B=4096, O=24, A=4, H=256,
               name="c4: synthetic obs=24 act=4 hidden=256, T=20 B=4096 (BASELINE.json configs[3])"),
    "c5": dict(T=100, B=8192, O=64, A=4, H=512,
               name="c5: long-unroll stress obs=64 act=4 (assumed, SURVEY 8) hidden=512, T=100 B=8192 (BASELINE.json configs[4])"),
}
WORKLOAD = {k: v for k, v in WORKLOADS["c4"].items() if k != "name"}
WORKLOAD_NAME = WORKLOADS["c4"]["name"]
METRIC = "learner steps/sec on synthetic (T=20,B=4096) trajectories"
SMS, FP32_LANES = 148, 128


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, on the process's original stdout."""
    out = _REAL_STDOUT or sys.__stdout__
    out.write(json.dumps(line) + "\n")
    out.flush()


def select_workload(cfg: str) -> None:
    global WORKLOAD, WORKLOAD_NAME, METRIC
    WORKLOAD = {k: v for k, v in WORKLOADS[cfg].items() if k != "name"}
    WORKLOAD_NAME = WORKLOADS[cfg]["name"]
    METRIC = f"learner steps/sec on synthetic (T={WORKLOAD['T']},B={WORKLOAD['B']}) trajectories"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=float(d["hbm_gbs"]), sm_max_mhz=float(d.get("sm_max_mhz", 1965.0)),
                    bf16_tflops=float(d.get("bf16_tflops", 1590.0)), source="MEASURED_PEAKS.json (measured)")
    return dict(hbm_gbs=6650.0, sm_max_mhz=1965.0, bf16_tflops=1590.0, source="fallback (B200_PROFILING.md)")


def hparams(B):
    from torched_impala_b200.utils import default_hparams

    return default_hparams(batch_size=B, max_timesteps=WORKLOAD["T"], policy_hidden_dims=WORKLOAD["H"],
                           value_fn_hidden_dims=WORKLOAD["H"])


# --------------------------------------------------------------------------- CPU baseline
class _TimedCounter:
    """utils.Counter stand-in (learner.py:254-255) that stamps the wall clock at every update."""

    def __init__(self):
        self.n, self.stamps = 0, [time.perf_counter()]

    def increment(self):
        self.n += 1
        self.stamps.append(time.perf_counter())

    @property
    def value(self):
        return self.n


def time_reference_learner(sample_B: int, warm: int, timed: int, threads: int):
    """The UNMODIFIED reference `Learner._learn` (learner.py:67-275) from oracle/_ref (or
    /root/reference), driven in-process through a list-backed queue; returns (median seconds per
    update, kind).  Falls back to the float64 per-trajectory port when the reference is absent."""
    import torch

    from oracle import refload
    from torched_impala_b200 import synth

    w = WORKLOAD
    torch.set_num_threads(threads)
    batch = synth.make_batch(1, w["T"], sample_B, w["O"], w["A"])
    trajs = synth.to_trajectories(batch)
    params = synth.init_params(0, w["O"], w["A"], w["H"])
    n = warm + timed
    if refload.available():
        ref_learner, ref_models, ref_utils = refload.load()
        hp = ref_utils.Hyperparameters(**hparams(sample_B)._replace(
            max_updates=n, eval_every=None, save_every=10 ** 9, verbose=0, log_path=None)._asdict())
        pol = ref_models.MlpPolicy(w["O"], w["A"], w["H"])
        vf = ref_models.MlpValueFn(w["O"], w["H"])
        for mod, grp in ((pol, "policy"), (vf, "value_fn")):
            mod.load_state_dict({k: torch.from_numpy(v).double() for k, v in params[grp].items()})
            mod.eval()  # the parity setting (SURVEY 0.4): Dropout(p=0.8) off
        cnt = _TimedCounter()
        lrn = ref_learner.Learner(1, hp, pol, vf, refload.ListQueue(trajs * n), cnt, None, timeout=1)
        cnt.stamps[0] = time.perf_counter()
        lrn._learn()
        times = [b - a for a, b in zip(cnt.stamps[:-1], cnt.stamps[1:])][warm:]
        kind = "reference"
    else:
        from oracle.cpu_learner_port import CpuLearnerPort

        port = CpuLearnerPort(params, hparams(sample_B), threads=threads)
        times = []
        for i in range(n):
            t0 = time.perf_counter()
            port.update(trajs)
            if i >= warm:
                times.append(time.perf_counter() - t0)
        kind = "port"
    return statistics.median(times), kind


def cpu_reference_numbers(warm: int, timed: int, budget_s: float = 120.0):
    """Times the reference CPU learner on this host.  Full batch when it fits `budget_s`, otherwise
    a bounded sample of trajectories scaled linearly (the reference loops over trajectories,
    learner.py:89: cost is linear in B) and labelled as such."""
    cores = os.cpu_count() or 1
    w = WORKLOAD
    probe_B = min(8, w["B"])  # tiny: with every host thread the per-trajectory python loop THRASHES (x100 slower)
    t1, kind = time_reference_learner(probe_B, 1, 1, 1)
    tn, _ = time_reference_learner(probe_B, 0, 1, cores) if cores > 1 else (t1, kind)
    threads, per_traj = (1, t1 / probe_B) if t1 <= tn else (cores, tn / probe_B)
    sample_B = w["B"]
    while sample_B > 64 and per_traj * sample_B * (warm + timed) > budget_s:
        sample_B //= 2
    t, kind = time_reference_learner(sample_B, warm, timed, threads)
    scale = w["B"] / sample_B
    from oracle import refload

    what = (f"the unmodified reference Learner._learn ({os.path.relpath(refload.reference_dir(), ROOT) if refload.reference_dir().startswith(ROOT) else refload.reference_dir()}, "
            "eval mode, in-process list queue)" if kind == "reference"
            else "oracle/cpu_learner_port.py (float64 per-trajectory port; reference modules not found)")
    return dict(value=1.0 / (t * scale), unit="steps/s", cores=threads, kind=kind, host_cores=cores,
                sample=(f"{what}: {warm}+{timed} updates of B={sample_B} (T={w['T']},O={w['O']},H={w['H']}), median"
                        + (f", scaled x{scale:g} to B={w['B']} (cost linear in B)" if scale != 1 else ", full batch")
                        + f"; probe at B={probe_B}: 1 thread {t1 * 1e3:.0f} ms, {cores} threads {tn * 1e3:.0f} ms per update"),
                sample_B=sample_B, timed_updates=timed, ms_per_update_sample=t * 1e3)


def reference_line(args, cb, steps, warm):
    w = WORKLOAD
    return dict(metric=METRIC, value=cb["value"], unit="steps/s", n_gpus=args.gpus, steps=steps,
                warmup=warm, ms_per_step=1e3 / cb["value"], higher_is_better=True, scaling="strong",
                vs_baseline=None, dtype="f64", data="synthetic", impl="reference",
                config=dict(workload=WORKLOAD_NAME, **w, global_batch=w["B"], per_gpu_batch=w["B"] // max(1, args.gpus)),
                cpu_baseline=cb,
                e2e=dict(value=cb["value"], unit="steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["CUDA_VISIBLE_DEVICES"] = ""  # the reference picks its device at import (learner.py:13)
    steps, warm = args.steps, max(1, min(args.warmup, 2))
    cb = cpu_reference_numbers(warm, steps)
    emit(reference_line(args, cb, steps, warm))


def learner_e2e(config: str, devices: int):
    """The same metric THROUGH the product API: forked `Learner(devices=N)` behind a `RingQueue` fed by
    32 synthetic actor processes (scripts/learner_e2e.py, fresh interpreter - this process has CUDA
    initialised and must not fork a CUDA child).  Includes queue -> slab packing in the actors, the
    per-rank shard DMAs, the update and the weight publication."""
    if config not in ("c3", "c4", "c5"):
        return None
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID"):
        env.pop(k, None)
    updates, warm = ("600", "100") if config != "c5" else ("200", "30")  # c5: 212 MB per update over PCIe
    cmd = [sys.executable, os.path.join(ROOT, "scripts", "learner_e2e.py"), "--config", config, "--actors", "32",
           "--updates", updates, "--warmup", warm, "--devices", str(devices), "--deadline", "90"]
    try:
        res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=240)
        for ln in reversed(res.stdout.splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return dict(error="no JSON line", stderr=res.stderr[-500:])
    except subprocess.TimeoutExpired:
        return dict(error="timed out")


def cpu_baseline(config: str):
    """`cpu_baseline` of the own arm: the reference arm in a fresh CPU-only subprocess (this process
    has CUDA initialised; the reference resolves its device at import), 1 + 3 updates."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    res = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--config", config,
                          "--steps", "3", "--warmup", "1"], capture_output=True, text=True, env=env, timeout=900)
    for ln in reversed(res.stdout.splitlines()):
        if ln.startswith("{"):
            return json.loads(ln)["cpu_baseline"]
    raise RuntimeError("cpu_baseline subprocess printed no JSON line:\n" + res.stderr[-2000:])


# --------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None
        # nvidia-smi needs a few hundred ms before its first line; wait so short runs get samples
        t_end = time.time() + 5.0
        while self.p is not None and time.time() < t_end and os.path.getsize(self.f.name) == 0:
            time.sleep(0.05)
        self.skip = 0

    def mark(self):
        """Discard everything sampled so far (idle clocks before the GPU is under load)."""
        self.f.flush()
        self.skip = os.path.getsize(self.f.name)

    def stop(self):
        if self.p is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(self.skip)
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.f.read().splitlines():
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for nm, val in zip(names, c[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        self.f.close()
        os.unlink(self.f.name)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons),
                    samples=len(sm))


# -------------------------------------------------------------------------------- own arm
def kernel_breakdown(eng, flush, iters=20, barrier=lambda: None):
    """CUDA-event time of every C-ABI launch of one step, eager, L2 flushed before each.

    N > 1 (push all-reduce): every rank runs the same call sequence; the backward is timed in its
    pushing variant (re-posting the current step's contribution is idempotent) and every timed
    optimizer call is preceded by an untimed stand-alone push, so its time includes the wait for
    the slowest peer's flag - the real cost of the exchange."""
    import ctypes as C

    import torch

    from torched_impala_b200 import _cabi
    from torched_impala_b200.engine import _ptr

    lib, hp, w = eng.lib, eng.hp, WORKLOAD
    T, B, O, A = eng.T, eng.B, eng.O, eng.A
    st = C.c_void_p(eng.stream.cuda_stream)
    p_pi = C.c_void_p(eng.params.data_ptr())
    p_vf = C.c_void_p(eng.params.data_ptr() + 4 * eng.n_pi)
    g_pi = C.c_void_p(eng.comm.data_ptr())
    g_vf = C.c_void_p(eng.comm.data_ptr() + 8 * eng.n_pi)
    scal = C.c_void_p(eng.comm.data_ptr() + 8 * eng.n_total)
    obs = _ptr(eng.d["obs"])
    calls = {
        "mlp_forward_pair(policy+value_fn)": lambda: lib.impala_mlp_forward_pair(
            obs, p_pi, p_vf, _ptr(eng.logits), _ptr(eng.values), eng.M_pi, eng.M_vf, O, eng.H_pi, eng.H_v, A, st),
        "mlp_backward_pair(policy+value_fn)": (lambda: lib.impala_mlp_backward_pair_push(
            obs, p_pi, p_vf, _ptr(eng.dlogits), _ptr(eng.dv), _ptr(eng.ws_pi), eng.ws_pi_bytes, _ptr(eng.ws_vf),
            eng.ws_vf_bytes, eng.M_pi, eng.M_vf, O, eng.H_pi, eng.H_v, A, scal, 4, _ptr(eng.peer["gather_ptrs"]),
            _ptr(eng.peer["seq"]), eng.peer["slot"], eng.peer["buf"], eng.peer["rank"], eng.world, st)) if (eng.peer and eng.peer["fused"]) else (lambda: lib.impala_mlp_backward_pair(
            obs, p_pi, p_vf, _ptr(eng.dlogits), _ptr(eng.dv), g_pi, g_vf, _ptr(eng.ws_pi), eng.ws_pi_bytes,
            _ptr(eng.ws_vf), eng.ws_vf_bytes, eng.M_pi, eng.M_vf, O, eng.H_pi, eng.H_v, A, st)),
        # the per-network entry points, for comparison (not launched by the step)
        "mlp_forward(policy)": lambda: lib.impala_mlp_forward(obs, p_pi, _ptr(eng.logits), eng.M_pi, O, eng.H_pi, A, st),
        "mlp_forward(value_fn)": lambda: lib.impala_mlp_forward(obs, p_vf, _ptr(eng.values), eng.M_vf, O, eng.H_v, 1, st),
        "vtrace_loss": lambda: lib.impala_vtrace_loss(
            _ptr(eng.logits), _ptr(eng.d["beh_logits"]), _ptr(eng.d["actions"]), _ptr(eng.d["rewards"]),
            _ptr(eng.d["done"]), _ptr(eng.d["lens"]), _ptr(eng.values), _ptr(eng.vs), _ptr(eng.pg_adv),
            _ptr(eng.dlogits), _ptr(eng.dv), scal, _ptr(eng.ws_vt), eng.ws_vt_bytes, T, B, A,
            float(hp.gamma), float(hp.rho_bar),
            float(hp.c_bar), float(hp.v_loss_c), float(hp.policy_loss_c), float(hp.entropy_c),
            float(eng.inv_batch), eng.mode, st),
        "mlp_backward(policy)": lambda: lib.impala_mlp_backward(obs, p_pi, _ptr(eng.dlogits), g_pi, _ptr(eng.ws_pi), eng.ws_pi_bytes, eng.M_pi, O, eng.H_pi, A, st),
        "mlp_backward(value_fn)": lambda: lib.impala_mlp_backward(obs, p_vf, _ptr(eng.dv), g_vf, _ptr(eng.ws_vf), eng.ws_vf_bytes, eng.M_vf, O, eng.H_v, 1, st),
    }
    H = eng.H_pi
    P = 2 * O * H + 3 * H + H * A + A + 1
    fl = {  # algorithmic FLOPs (SURVEY.md 8d: no recompute counted)
        "mlp_forward(policy)": 2.0 * eng.M_pi * (O * H + H * A),
        "mlp_forward(value_fn)": 2.0 * eng.M_vf * (O * eng.H_v + eng.H_v),
        "mlp_backward(policy)": 2.0 * eng.M_pi * (O * H + 2 * H * A),
        "mlp_backward(value_fn)": 2.0 * eng.M_vf * (O * eng.H_v + 2 * eng.H_v),
    }
    fl["mlp_forward_pair(policy+value_fn)"] = fl["mlp_forward(policy)"] + fl["mlp_forward(value_fn)"]
    fl["mlp_backward_pair(policy+value_fn)"] = fl["mlp_backward(policy)"] + fl["mlp_backward(value_fn)"]
    by = {  # algorithmic bytes of the HBM-bound kernels
        # in: cur+beh logits, actions, rewards, done, v ; out: vs, pg_adv, dlogits, dv
        "vtrace_loss": 4.0 * T * B * (2 * A + 2) + T * B + 4.0 * (T + 1) * B
                       + 4.0 * (T + 1) * B + 4.0 * T * B + 4.0 * T * B * A + 4.0 * (T + 1) * B,
    }
    out = {}
    with torch.cuda.stream(eng.stream):
        for name, fn in calls.items():
            barrier()
            ts = []
            for _ in range(iters):
                flush()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(eng.stream)
                _cabi.check(fn(), name)
                e1.record(eng.stream)
                e1.synchronize()
                ts.append(e0.elapsed_time(e1) * 1e3)
            out[name] = dict(us=statistics.median(ts), flops=fl.get(name), bytes=by.get(name))
        # stand-alone V-trace scan at the long-unroll stress shape (BASELINE configs[4]: T=100,
        # B=8192, A=4): the one kernel of the path that is genuinely HBM-bandwidth bound
        Tl, Bl2, Al = 100, 8192, 4
        g = torch.Generator(device=eng.dev).manual_seed(0)
        cur = torch.randn(Tl, Bl2, Al, device=eng.dev, generator=g)
        beh = torch.randn(Tl, Bl2, Al, device=eng.dev, generator=g)
        act = torch.randint(0, Al, (Tl, Bl2), device=eng.dev, generator=g, dtype=torch.int32)
        rew = torch.randn(Tl, Bl2, device=eng.dev, generator=g)
        don = torch.zeros(Tl, Bl2, dtype=torch.uint8, device=eng.dev)
        lens_l = torch.full((Bl2,), Tl, dtype=torch.int32, device=eng.dev)
        vv = torch.randn(Tl + 1, Bl2, device=eng.dev, generator=g)
        vs_o = torch.empty(Tl + 1, Bl2, device=eng.dev)
        pg_o = torch.empty(Tl, Bl2, device=eng.dev)
        ts = []
        for _ in range(iters):
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(eng.stream)
            _cabi.check(lib.impala_vtrace(_ptr(cur), _ptr(beh), _ptr(act), _ptr(rew), _ptr(don), _ptr(lens_l),
                                          _ptr(vv), _ptr(vs_o), _ptr(pg_o), Tl, Bl2, Al, float(hp.gamma),
                                          float(hp.rho_bar), float(hp.c_bar), eng.mode, st), "impala_vtrace")
            e1.record(eng.stream)
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        # SURVEY 8d: 4TB(2A+2) + TB + 4(T+1)B in, 4(T+1)B + 4TB out = 43 483 136 B
        out["vtrace(T=100,B=8192 stand-alone)"] = dict(
            us=statistics.median(ts), flops=None,
            bytes=4.0 * Tl * Bl2 * (2 * Al + 2) + Tl * Bl2 + 4.0 * (Tl + 1) * Bl2 + 4.0 * (Tl + 1) * Bl2 + 4.0 * Tl * Bl2)
        del cur, beh, act, rew, don, lens_l, vv, vs_o, pg_o
        # optimizer: needs a valid gradient in comm; time it on copies so parameters stay intact
        barrier()
        ts, ts_push = [], []
        keep = [t.clone() for t in (eng.params, eng.adam_m, eng.adam_v, eng.adam_step)]
        pr = eng.peer
        for _ in range(iters):
            flush()
            if pr:  # this step's contribution -> every rank (stand-alone producer), timed on its own
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(eng.stream)
                _cabi.check(lib.impala_peer_push(_ptr(eng.comm), eng.n_total + 8, _ptr(pr["gather_ptrs"]), _ptr(pr["seq"]),
                                                 pr["slot"], pr["buf"], pr["rank"], eng.world, st), "impala_peer_push")
                e1.record(eng.stream)
                ts_push.append((e0, e1))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(eng.stream)
            eng._enqueue_opt()
            e1.record(eng.stream)
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        for dst, src in zip((eng.params, eng.adam_m, eng.adam_v, eng.adam_step), keep):
            dst.copy_(src)
        # read grad (N = 1: f64; N > 1: `world` local 16-byte LL elements per entry) + params/m/v rw
        out["gather+clip_adam" if pr else "clip_adam"] = dict(
            us=statistics.median(ts), flops=None, bytes=((16.0 * eng.world if pr else 8.0) + 6 * 4.0) * eng.n_total)
        if pr:
            out["peer_push(stand-alone)"] = dict(us=statistics.median([a.elapsed_time(b) * 1e3 for a, b in ts_push]),
                                                 flops=None, bytes=16.0 * eng.world * (eng.n_total + 8))
    eng.synchronize()
    return out


DUMP_LIMIT = 64 << 20  # bytes, all arrays of one --dump-outputs together


def last_step_outputs(eng, scalars):
    """What the last timed step hands its caller, as float32 / float64 numpy arrays: the logged loss
    scalars, the V-trace targets and advantages of this rank's batch, the gradient of the step
    (float64, before clipping) and both networks' parameters after the update."""
    import numpy as np
    import torch

    eng.synchronize()
    out = {"scalars": np.array([scalars[k] for k in ("value_fn_loss", "policy_loss", "policy_entropy", "total_loss",
                                                     "batch_mean_reward")], np.float64),
           "vs": eng.vs.cpu().numpy(), "pg_adv": eng.pg_adv.cpu().numpy()}
    for g, sd in eng.state(torch.float32).items():
        for k, v in sd.items():
            out[f"params.{g}.{k}"] = v.numpy()
    for g, sd in eng.grads().items():
        for k, v in sd.items():
            out[f"grad.{g}.{k}"] = v
    assert sum(v.nbytes for v in out.values()) == dump_bytes(eng)  # the size checked before the run
    return out


def dump_bytes(eng) -> int:
    """Size of last_step_outputs(eng): 5 float64 scalars, vs + pg_adv (float32), params (float32) + grad (float64)."""
    n_params = sum(math.prod(shp) for _, _, _, shp in eng._segments())
    return 8 * 5 + 4 * (eng.vs.numel() + eng.pg_adv.numel()) + (4 + 8) * n_params


def dump_outputs(path, outputs):
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for name, v in outputs.items():
        np.save(os.path.join(path, name + ".npy"), v)


def run_own_arm(args):
    import torch

    from torched_impala_b200 import synth
    from torched_impala_b200.engine import LearnerEngine

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the learner has no CPU path)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch with torchrun")
    torch.cuda.set_device(local)
    pg = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        pg = dist.group.WORLD
    w = WORKLOAD
    Bl = w["B"] // world
    hp = hparams(w["B"])
    eng = LearnerEngine(w["T"], Bl, w["O"], w["A"], w["H"], w["H"], hp, global_batch=w["B"],
                        device=f"cuda:{local}", process_group=pg, use_graph=not args.no_graph)
    if args.dump_outputs and dump_bytes(eng) > DUMP_LIMIT:
        raise SystemExit(f"bench.py: --dump-outputs would write {dump_bytes(eng)} bytes, more than {DUMP_LIMIT}")
    params0 = synth.init_params(0, w["O"], w["A"], w["H"])
    batches = [synth.shard_batch(synth.make_batch(1 + i, w["T"], w["B"], w["O"], w["A"]), rank, world)
               for i in range(2)]
    # ---------------- parity of this very configuration (checker, outside every timed region):
    # one step from the initial parameters on batch 0 against the float64 oracle (oracle/check.py);
    # with N ranks every rank checks its shard and the oracle sums are all-reduced.
    parity = None
    if not args.no_parity:
        from oracle.check import first_step_parity

        t_par = time.perf_counter()
        parity = first_step_parity(eng, params0, batches[0], group=pg)
        parity["seconds"] = round(time.perf_counter() - t_par, 2)
    eng.load_state(params0)
    for i, b in enumerate(batches):
        eng.fill_host(b, i)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=eng.dev)  # 2x the 126 MB L2

    def flush():
        flush_buf.zero_()  # on the current (= engine) stream

    def barrier():
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        import torch.distributed as dist

        t = torch.tensor([x], dtype=torch.float64, device=eng.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-resident ("value") ----------------
    eng.ingest(0)
    eng.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    with torch.cuda.stream(eng.stream):
        for i in range(max(3, args.warmup)):
            flush()
            eng.step()
            if i == 0 and sampler:
                torch.cuda.synchronize()
                sampler.mark()  # clocks are sampled from here to the end of the e2e loop
    barrier()
    evs = []
    with torch.cuda.stream(eng.stream):
        for _ in range(args.steps):
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(eng.stream)
            eng.step()
            e1.record(eng.stream)
            evs.append((e0, e1))
    barrier()
    dev_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in evs))
    launches = eng.launches_per_step * args.steps
    scal_dev = eng.read_scalars()
    outputs = last_step_outputs(eng, scal_dev) if args.dump_outputs and rank == 0 else None

    # ---------------- end to end through host buffers ----------------
    # software pipeline: the DMA of batch i+1 (copy stream) runs under the kernels of batch i;
    # the host reads step i-1's scalars while step i runs.  Every step's H2D and D2H happen
    # inside the timed region.
    def e2e_loop(n):
        last = None
        eng.ingest(0)
        prev = None
        for i in range(n):
            if i + 1 < n:
                eng.ingest((i + 1) % 2)   # H2D of the next step's inputs from pinned memory
            eng.step(i % 2)
            tk = eng.post_scalars()       # D2H of this step's loss scalars
            if prev is not None:
                last = eng.fetch_scalars(prev)
            prev = tk
        last = eng.fetch_scalars(prev)
        eng.synchronize()
        return last

    e2e_loop(max(3, args.warmup))
    barrier()
    t0 = time.perf_counter()
    e_start, e_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_start.record(eng.stream)
    last = e2e_loop(args.steps)
    e_stop.record(eng.stream)
    barrier()
    e2e_wall_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    e2e_dev_ms = max_over_ranks(e_start.elapsed_time(e_stop))
    clock_note = None
    if dev_ms + e2e_dev_ms < 80.0:
        # nvidia-smi samples every 20 ms: short runs (small --steps) would end without a single
        # sample under load.  Keep the same step loop running (untimed, every rank the same count -
        # the multi-GPU optimizer kernel is a collective) until ~100 ms are covered.
        n_probe = int(100.0 / max(dev_ms / args.steps, 1e-3)) + 1
        with torch.cuda.stream(eng.stream):
            for i in range(n_probe):
                eng.step()
                if i % 256 == 255:
                    eng.synchronize()
        eng.synchronize()
        clock_note = (f"timed regions covered {dev_ms + e2e_dev_ms:.1f} ms, less than a few 20 ms nvidia-smi periods: "
                      f"sampling continued over {n_probe} more (untimed) steps of the same loop")
    clocks = sampler.stop() if sampler else None
    if clocks is not None and clock_note:
        clocks["note"] = clock_note

    # ---------------- per-kernel roofline (rank 0 reports) ----------------
    with torch.cuda.stream(eng.stream):
        kern = kernel_breakdown(eng, flush, barrier=barrier)
    pk = peaks()
    fp32_peak = SMS * FP32_LANES * 2 * pk["sm_max_mhz"] * 1e6 / 1e12  # TFLOP/s at max SM clock
    tf32_peak = pk["bf16_tflops"] / 2.0  # tf32 UMMA rate = half the (measured) bf16 rate
    H, O, A = eng.H_pi, eng.O, eng.A
    tc_on = os.environ.get("IMPALA_MLP_TC", "1") != "0" and O % 4 == 0 and A <= 4
    narrow = tc_on and 4 <= O <= 28 and H in (128, 256)                       # mlp_fwd_tc.cu / mlp_bwd_tc.cu
    wide = (tc_on and not narrow and 4 <= O <= 64 and H % 128 == 0 and H <= 4096
            and os.environ.get("IMPALA_MLP_TCW", "1") != "0")                 # mlp_tcw.cu (c5)
    on_tc = narrow or wide
    # tensor-core work actually issued: 3xTF32 (3 UMMAs per product).  Narrow kernels: forward and recompute
    # K = [x | 1] padded to a multiple of 8, dW1 reduction over 32 output columns.  Wide kernels: K = O
    # padded to 8 (the bias is added on the CUDA cores), dW1 reduction over 64 output columns.
    kb = (O + 7) // 8 * 8
    kf, ncol = ((O + 1 + 7) // 8 * 8, 32) if narrow else (kb, 64)
    executed = {"mlp_forward(policy)": 2.0 * eng.M_pi * H * kf * 3, "mlp_forward(value_fn)": 2.0 * eng.M_vf * H * kf * 3,
                "mlp_backward(policy)": 2.0 * eng.M_pi * H * (kf + ncol) * 3,
                "mlp_backward(value_fn)": 2.0 * eng.M_vf * H * (kf + ncol) * 3}
    executed["mlp_forward_pair(policy+value_fn)"] = executed["mlp_forward(policy)"] + executed["mlp_forward(value_fn)"]
    executed["mlp_backward_pair(policy+value_fn)"] = executed["mlp_backward(policy)"] + executed["mlp_backward(value_fn)"]
    kernels = {}
    for name, k in kern.items():
        ent = dict(us=round(k["us"], 3))
        if k["flops"]:
            ach = k["flops"] / (k["us"] * 1e-6) / 1e12
            if on_tc:
                ex = executed[name] / (k["us"] * 1e-6) / 1e12
                ent.update(bound="tensor", achieved=round(ach, 3), peak=round(tf32_peak, 1), unit="TFLOP/s",
                           frac=round(ach / tf32_peak, 4), executed_tflops=round(ex, 1),
                           executed_frac=round(ex / tf32_peak, 4))
            else:
                ent.update(bound="fp32", achieved=round(ach, 3), peak=round(fp32_peak, 2), unit="TFLOP/s",
                           frac=round(ach / fp32_peak, 4))
        else:
            ach = k["bytes"] / (k["us"] * 1e-6) / 1e9
            ent.update(bound="hbm", achieved=round(ach, 1), peak=pk["hbm_gbs"], unit="GB/s",
                       frac=round(ach / pk["hbm_gbs"], 4))
        kernels[name] = ent
    in_step = ("mlp_forward_pair(policy+value_fn)", "vtrace_loss", "mlp_backward_pair(policy+value_fn)",
               "gather+clip_adam" if eng.peer else "clip_adam")
    for n in kernels:
        kernels[n]["in_step"] = n in in_step
    dom = max(in_step, key=lambda n: kernels[n]["us"])
    traffic = None
    # ncu dram__bytes per launch of the dominant kernel: profiles/dram_traffic.json is the c4 capture,
    # other configs have their own file (dram_traffic_c5.json) or report null
    prof = os.path.join(ROOT, "profiles", "dram_traffic.json" if args.config == "c4" else f"dram_traffic_{args.config}.json")
    if os.path.exists(prof):
        with open(prof) as f:
            traffic = json.load(f).get(dom)
    src = {"hbm": pk["source"],
           "tensor": f"tf32 UMMA peak = measured bf16 {pk['bf16_tflops']:.1f} TF/s / 2 ({pk['source']}); `achieved` counts "
                     "ALGORITHMIC fp32 FLOPs (SURVEY 8d), `executed_tflops` the 3xTF32 / K-padded / recompute work issued",
           "fp32": f"148 SMs x 128 FP32 lanes x 2 x {pk['sm_max_mhz']:.0f} MHz (max SM clock, {pk['source']}); "
                   "MEASURED_PEAKS has no FP32 figure"}[kernels[dom]["bound"]]
    roofline = dict(kernel=dom, traffic=traffic, peak_source=src,
                    **{k: kernels[dom][k] for k in kernels[dom] if k not in ("us", "in_step")})

    # ---------------- weak scaling beside the strong line: B per GPU = the full workload batch
    weak = None
    if world > 1 and not args.no_weak:
        hp_w = hparams(w["B"] * world)
        eng_w = LearnerEngine(w["T"], w["B"], w["O"], w["A"], w["H"], w["H"], hp_w, global_batch=w["B"] * world,
                              device=f"cuda:{local}", process_group=pg, use_graph=not args.no_graph)
        eng_w.load_state(params0)
        eng_w.load_device_batch(synth.make_batch(100 + rank, w["T"], w["B"], w["O"], w["A"]))
        with torch.cuda.stream(eng_w.stream):
            for _ in range(max(3, args.warmup)):
                flush()
                eng_w.step()
        barrier()
        evw = []
        with torch.cuda.stream(eng_w.stream):
            for _ in range(args.steps):
                flush()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(eng_w.stream)
                eng_w.step()
                e1.record(eng_w.stream)
                evw.append((e0, e1))
        barrier()
        ms_w = max_over_ranks(sum(a.elapsed_time(b) for a, b in evw)) / args.steps
        weak = dict(scaling="weak", per_gpu_batch=w["B"], global_batch=w["B"] * world, ms_per_step=ms_w,
                    steps_per_s=1e3 / ms_w, trajectories_per_s=1e3 / ms_w * w["B"] * world,
                    note="same step with B per GPU = the workload's full batch; value of the line stays the strong-scaling number")
        del eng_w
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    if rank != 0:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()
        return
    cb = cpu_baseline(args.config) if world == 1 and not args.no_cpu else None
    e2e_learner = learner_e2e(args.config, world) if not args.no_learner else None
    ms = dev_ms / args.steps
    line = dict(
        metric=METRIC, value=1e3 / ms, unit="steps/s", n_gpus=world, steps=args.steps,
        warmup=max(3, args.warmup), ms_per_step=ms, higher_is_better=True, scaling="strong",
        vs_baseline=None, dtype="f32", data="synthetic",
        config=dict(workload=WORKLOAD_NAME, **w, global_batch=w["B"], per_gpu_batch=Bl,
                    parallelism=f"dp{world} (batch sharded, 1 all-reduce of {8 * (eng.n_total + 8)} B/step (16-byte LL elements on the wire), "
                                f"{('pushed over NVLink peer memory from the ' + ('backward kernel tail' if eng.peer['fused'] else 'stand-alone producer kernel')) if eng.peer else 'NCCL'})"
                    if world > 1 else "single GPU",
                    l2="flushed between timed steps (256 MiB memset on the launching stream)",
                    cuda_graph=not args.no_graph, timing="sum of per-step CUDA-event intervals, max over ranks"),
        clocks=clocks, gpu_launches=launches,
        e2e=dict(value=args.steps / (e2e_wall_ms * 1e-3), unit="steps/s",
                 h2d_bytes_per_step=int(eng.slab_bytes) * world, d2h_bytes_per_step=48 * world,
                 ms_per_step_wall=e2e_wall_ms / args.steps, ms_per_step_device=e2e_dev_ms / args.steps,
                 note=("wall clock around K x (H2D from pinned slab, step, D2H of scalars), max over ranks; "
                       "copy of batch i+1 overlaps compute of batch i (double-buffered slabs)")),
        roofline=roofline, kernels=kernels,
        loss=dict(device_resident=scal_dev["total_loss"], e2e_last=last["total_loss"]),
        parity=parity,
    )
    if weak:
        line["weak_scaling"] = weak
    if e2e_learner:
        line["e2e_learner"] = e2e_learner
    if cb:
        line["cpu_baseline"] = cb
    if outputs:
        dump_outputs(args.dump_outputs, outputs)
    emit(line)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


def positive_int(s: str) -> int:
    if int(s) < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {s}")
    return int(s)


def main():
    # Libraries (NCCL prints its version banner) may write to stdout; the contract is ONE JSON
    # line there.  Keep the real stdout aside, point fd 1 at stderr for the duration of the run
    # and emit the JSON line through the saved descriptor.
    global _REAL_STDOUT
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr  # python-level prints (the reference learner is chatty) go to stderr too
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=200, help="timed steps")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA graphs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--config", default="c4", choices=sorted(WORKLOADS), help="BASELINE.json config (default: c4, the metric's)")
    ap.add_argument("--no-parity", action="store_true", help="skip the first-step oracle check")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the weak-scaling measurement")
    ap.add_argument("--no-learner", action="store_true", help="skip the run through Learner + RingQueue + actor processes")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, to compare builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 arm's timed steps")
    select_workload(args.config)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_own_arm(args)
    _REAL_STDOUT.flush()


if __name__ == "__main__":
    main()
