"""Host-side step engine of the B200 learner: buffers, streams, CUDA graph, peer buffers.

One `LearnerEngine` lives in the learner process of one GPU.  It owns every device
buffer of the update path and enqueues, per learner step, exactly the C-ABI calls of
include/impala_b200.h (PyTorch only provides device memory, streams and
`torch.distributed`):

    impala_ingest              pinned host slab -> device slab (one DMA)        learner.py:104-109,117
    impala_mlp_forward_pair    policy logits (T*B rows) + values ((T+1)*B)      learner.py:112-113
    impala_vtrace_loss         V-trace, 3 losses, dL/dlogits, dL/dv, scalars    learner.py:116-162
    impala_mlp_backward_pair   parameter gradients of both nets (float64)       learner.py:175
    impala_clip_adam           per-net clip + Adam + step counter               learner.py:176-183
      N > 1 (new; SURVEY 8e): the all-reduce of [grads | scalars] is a PUSH over NVLink peer memory -
      the tail of impala_mlp_backward_pair_push (or impala_peer_push for shapes it does not cover)
      stores this rank's contribution, every value tagged with the step number (LL format), into
      every rank's gather buffer; impala_gather_clip_adam polls its local slots, adds them in rank
      order and applies the update.  IMPALA_ALLREDUCE=nccl: torch.distributed all-reduce between the
      backward and impala_clip_adam instead.

With `use_graph=True` the whole launch sequence of a step is captured once per slab into ONE CUDA
graph and replayed (two graphs around the collective in the NCCL scheme).
Ingest is double buffered: two pinned host slabs, two device slabs and
a dedicated copy stream, so the DMA of batch i+1 runs under the kernels of batch i
(`ingest(slot)` / `step(slot)` order themselves with events); the loss scalars come back
through a small ring of pinned buffers (`post_scalars` / `fetch_scalars`) so the host only
ever waits for the previous step.
"""
from __future__ import annotations

import contextlib
import ctypes as C

import numpy as np
import torch

from . import _cabi

PKEYS = ("model.0.weight", "model.0.bias", "model.3.weight", "model.3.bias")
SCALAR_NAMES = ("value_fn_loss", "policy_loss", "policy_entropy", "batch_mean_reward")
_BATCH_FIELDS = (("obs", np.float32), ("beh_logits", np.float32), ("actions", np.int32),
                 ("rewards", np.float32), ("done", np.uint8), ("lens", np.int32))
_TORCH_DT = {np.float32: torch.float32, np.int32: torch.int32, np.uint8: torch.uint8}


def _ptr(t: torch.Tensor) -> C.c_void_p:
    return C.c_void_p(t.data_ptr())


class LearnerEngine:
    def __init__(self, T: int, B_local: int, O: int, A: int, H_pi: int, H_v: int, hp,
                 global_batch: int | None = None, device: str | torch.device = "cuda:0",
                 mode: str = "reference", process_group=None, use_graph: bool = True,
                 slabs: int = 2):
        if not torch.cuda.is_available():
            raise _cabi.ImpalaCudaError("LearnerEngine needs a CUDA device; there is no CPU path")
        self.lib = _cabi.lib()
        self.dev = torch.device(device)
        torch.cuda.set_device(self.dev)
        self.T, self.B, self.O, self.A, self.H_pi, self.H_v = T, B_local, O, A, H_pi, H_v
        self.hp = hp
        self.mode = _cabi.MODES[mode]
        self.pg = process_group
        self.world = 1
        if process_group is not None:
            import torch.distributed as dist

            self.world = dist.get_world_size(process_group)
        self.global_batch = int(global_batch if global_batch is not None else B_local * self.world)
        self.inv_batch = 1.0 / self.global_batch
        self.use_graph = use_graph
        self.stream = torch.cuda.Stream(device=self.dev)
        self.copy_stream = torch.cuda.Stream(device=self.dev)
        self.launches_per_step = 0

        # ---- parameter blocks: [policy | value_fn], float32, 128-byte aligned tensors
        self.pi_off, self.n_pi = _cabi.param_layout(O, H_pi, A)
        self.vf_off, self.n_vf = _cabi.param_layout(O, H_v, 1)
        self.n_total = self.n_pi + self.n_vf
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.params = torch.zeros(self.n_total, **f32)
        self.adam_m = torch.zeros(self.n_total, **f32)
        self.adam_v = torch.zeros(self.n_total, **f32)
        self.adam_step = torch.zeros(3, dtype=torch.int64, device=self.dev)  # step, beta1^t, beta2^t bits
        # float64 [gradient | 4 loss scalars | pad]: the all-reduce payload
        self.comm = torch.zeros(self.n_total + 8, dtype=torch.float64, device=self.dev)
        self.norms = torch.zeros(2, dtype=torch.float64, device=self.dev)

        # ---- batch slab (device) and pinned staging slabs (host), identical layouts
        self.slab_off, self.slab_bytes = _cabi.batch_layout(T, B_local, O, A)
        self.n_slabs = slabs
        self.d_slabs = [torch.zeros(self.slab_bytes, dtype=torch.uint8, device=self.dev)
                        for _ in range(slabs)]
        self.h_slabs = [torch.zeros(self.slab_bytes, dtype=torch.uint8).pin_memory()
                        for _ in range(slabs)]
        shapes = {"obs": (T + 1, B_local, O), "beh_logits": (T, B_local, A),
                  "actions": (T, B_local), "rewards": (T, B_local), "done": (T, B_local),
                  "lens": (B_local,)}
        self.shapes = shapes
        self.d_views, self.h_views = [], []
        for dslab, hslab in zip(self.d_slabs, self.h_slabs):
            arr = hslab.numpy()
            dv, hv = {}, {}
            for (name, dt), off in zip(_BATCH_FIELDS, self.slab_off):
                n = int(np.prod(shapes[name])) * np.dtype(dt).itemsize
                dv[name] = dslab[off:off + n].view(_TORCH_DT[dt]).view(shapes[name])
                hv[name] = arr[off:off + n].view(dt).reshape(shapes[name])
            self.d_views.append(dv)
            self.h_views.append(hv)
        self.d = self.d_views[0]
        self.slab_ready = [torch.cuda.Event() for _ in range(slabs)]  # H2D into slab done
        self.slab_free = [torch.cuda.Event() for _ in range(slabs)]   # last consumer of slab done
        self._slab_used = [False] * slabs

        # ---- activations / gradients of the non-MLP part
        self.logits = torch.zeros(T, B_local, A, **f32)
        self.values = torch.zeros(T + 1, B_local, **f32)
        self.vs = torch.zeros(T + 1, B_local, **f32)
        self.pg_adv = torch.zeros(T, B_local, **f32)
        self.dlogits = torch.zeros(T, B_local, A, **f32)
        self.dv = torch.zeros(T + 1, B_local, **f32)
        self.M_pi, self.M_vf = T * B_local, (T + 1) * B_local
        self.ws_pi_bytes = self._ws_bytes(self.M_pi, O, H_pi, A)
        self.ws_vf_bytes = self._ws_bytes(self.M_vf, O, H_v, 1)
        self.ws_pi = torch.zeros(self.ws_pi_bytes, dtype=torch.uint8, device=self.dev)
        self.ws_vf = torch.zeros(self.ws_vf_bytes, dtype=torch.uint8, device=self.dev)
        self.ws_vt_bytes = int(self.lib.impala_vtrace_loss_workspace(T, B_local, A))
        self.ws_vt = torch.zeros(self.ws_vt_bytes, dtype=torch.uint8, device=self.dev)  # zeroed once
        self.h_scalars = torch.zeros(4, 8, dtype=torch.float64).pin_memory()  # ring of 4 tickets
        self._scalar_events = [torch.cuda.Event() for _ in range(4)]
        self._ticket = 0

        self._loop_thread = None  # thread whose current stream IS self.stream for a whole update loop (loop_stream)
        self._graph_main = {}  # slab slot -> captured step
        self._graph_opt = None
        self._main_launches = 0
        self.steps_done = 0
        self.peer = None
        if self.world > 1:
            self._setup_peer_allreduce()

    # ------------------------------------------------------------------ parameters
    # ------------------------------------------------------------------------ multi-GPU plumbing
    def _setup_peer_allreduce(self) -> None:
        """Allocate this rank's gather buffer (LL elements, 16 bytes per float64) and map every peer's
        (CUDA IPC over NVLink) for the push-model all-reduce.  IMPALA_ALLREDUCE=nccl - or a failed mapping on ANY rank -
        keeps the torch.distributed all-reduce between the backward and the optimizer instead."""
        import os
        import warnings

        import torch.distributed as dist

        rank, world = dist.get_rank(self.pg), self.world
        ok, err, mine = os.environ.get("IMPALA_ALLREDUCE", "peer") != "nccl" and world <= 8, "", {}
        lib = self.lib
        slot = self.n_total + 8                         # LL elements per rank slot: [gradient | scalars | pad]
        buf = world * slot                              # LL elements per parity buffer
        if ok:
            try:
                ptr, handle = C.c_void_p(), (C.c_char * 64)()
                _cabi.check(lib.impala_peer_alloc(2 * 16 * buf, C.byref(ptr), handle), "impala_peer_alloc")
                mine["gather"] = (ptr.value, bytes(handle.raw))
            except Exception as e:  # noqa: BLE001 - reported below, all ranks fall back together
                ok, err = False, repr(e)
        handles = [None] * world
        dist.all_gather_object(handles, {k: v[1] for k, v in mine.items()} if ok else None, group=self.pg)
        ok = ok and all(h is not None for h in handles)
        gather_ptrs, opened = [], []
        if ok:
            try:
                for r, h in enumerate(handles):
                    if r == rank:
                        gather_ptrs.append(mine["gather"][0])
                    else:
                        ptr = C.c_void_p()
                        _cabi.check(lib.impala_peer_open(h["gather"], C.byref(ptr)), f"impala_peer_open(rank {r})")
                        opened.append(ptr.value)
                        gather_ptrs.append(ptr.value)
            except Exception as e:  # noqa: BLE001
                ok, err = False, repr(e)
        agree = torch.tensor([1 if ok else 0], device=self.dev)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN, group=self.pg)
        if int(agree.item()) == 0:
            if os.environ.get("IMPALA_ALLREDUCE", "peer") != "nccl" and rank == 0:
                warnings.warn(f"peer-memory all-reduce unavailable ({err or 'a rank could not map its peers'}); "
                              "using the NCCL all-reduce between backward and optimizer")
            return
        i64 = dict(dtype=torch.int64, device=self.dev)
        fused = bool(lib.impala_mlp_backward_pair_push_supported(self.M_pi, self.M_vf, self.O, self.H_pi, self.H_v, self.A))
        self.peer = dict(gather=mine["gather"][0], opened=opened, gather_ptrs=torch.tensor(gather_ptrs, **i64),
                         seq=torch.zeros(1, **i64), rank=rank, slot=slot, buf=buf, fused=fused,
                         err=torch.zeros(1, dtype=torch.int32, device=self.dev),
                         timeout_s=float(os.environ.get("IMPALA_PEER_TIMEOUT_S", "600")))
        torch.cuda.synchronize(self.dev)
        dist.barrier(group=self.pg)

    def _ws_bytes(self, M, O, H, N2):
        n = self.lib.impala_mlp_backward_workspace(M, O, H, N2)
        if n < 0:
            _cabi.check(int(n), f"impala_mlp_backward_workspace(M={M},O={O},H={H},N2={N2})")
        return int(n)

    def _segments(self):
        """(group, key, flat offset, shape) of every parameter tensor in `self.params`."""
        O, A = self.O, self.A
        shp_pi = ((self.H_pi, O), (self.H_pi,), (A, self.H_pi), (A,))
        shp_vf = ((self.H_v, O), (self.H_v,), (1, self.H_v), (1,))
        for key, off, shp in zip(PKEYS, self.pi_off, shp_pi):
            yield "policy", key, off, shp
        for key, off, shp in zip(PKEYS, self.vf_off, shp_vf):
            yield "value_fn", key, self.n_pi + off, shp

    def load_state(self, state: dict) -> None:
        """state = {"policy": state_dict, "value_fn": state_dict} (any float dtype, CPU)."""
        flat = torch.zeros(self.n_total, dtype=torch.float32)
        for grp, key, off, shp in self._segments():
            t = torch.as_tensor(np.asarray(state[grp][key]) if not torch.is_tensor(state[grp][key])
                                else state[grp][key].detach().cpu())
            if tuple(t.shape) != tuple(shp):
                raise ValueError(f"{grp}.{key}: expected {shp}, got {tuple(t.shape)}")
            flat[off:off + t.numel()] = t.reshape(-1).to(torch.float32)
        self.params.copy_(flat)
        torch.cuda.synchronize(self.dev)

    def state(self, dtype=torch.float64) -> dict:
        """Reference-format state_dicts (CPU, float64 like reference models.py:6)."""
        self.stream.synchronize()
        flat = self.params.detach().cpu()
        out = {"policy": {}, "value_fn": {}}
        for grp, key, off, shp in self._segments():
            n = int(np.prod(shp))
            out[grp][key] = flat[off:off + n].reshape(shp).to(dtype).clone()
        return out

    def grads(self) -> dict:
        """Last step's pre-clip gradient (float64), reference state_dict layout."""
        self.stream.synchronize()
        flat = self.comm[: self.n_total].detach().cpu()
        out = {"policy": {}, "value_fn": {}}
        for grp, key, off, shp in self._segments():
            n = int(np.prod(shp))
            out[grp][key] = flat[off:off + n].reshape(shp).numpy().copy()
        return out

    # ---------------------------------------------------------------------- ingest
    def host_batch(self, slot: int = 0) -> dict:
        """Writable numpy views of pinned staging slab `slot` (fill these, then ingest)."""
        return self.h_views[slot]

    def fill_host(self, batch: dict, slot: int = 0) -> None:
        for name, _ in _BATCH_FIELDS:
            np.copyto(self.h_views[slot][name], batch[name])

    def _copy_to_slab(self, slot: int, fn: str, *args) -> None:
        """lib.<fn>(device slab `slot`, *args, copy stream), ordered after the step that last read the slab."""
        cs = self.copy_stream
        if self._slab_used[slot]:
            cs.wait_event(self.slab_free[slot])
        _cabi.check(getattr(self.lib, fn)(_ptr(self.d_slabs[slot]), *args, C.c_void_p(cs.cuda_stream)), fn)
        self.slab_ready[slot].record(cs)

    def ingest(self, slot: int = 0) -> None:
        """Async H2D of pinned slab `slot` into device slab `slot` on the copy stream."""
        self.ingest_from(self.h_slabs[slot].data_ptr(), slot)

    def register_host(self, address: int, nbytes: int) -> None:
        """Page-lock caller-owned host memory (e.g. a shared-memory trajectory ring) for DMA."""
        rc = torch.cuda.cudart().cudaHostRegister(address, nbytes, 0)
        if int(rc) != 0:
            raise _cabi.ImpalaCudaError(f"cudaHostRegister failed: {rc}")

    def ingest_from(self, host_address: int, slot: int = 0) -> None:
        """Like `ingest`, but the source slab is caller-owned (registered) host memory in the
        same batch layout - the DMA reads the actors' shared-memory slab directly."""
        self._copy_to_slab(slot, "impala_ingest", C.c_void_p(host_address), self.slab_bytes)

    def ingest_shard_from(self, host_address: int, b0: int, B_total: int, slot: int = 0) -> None:
        """Data-parallel ingest: columns [b0, b0 + B_local) of a caller-owned (registered) host slab
        laid out for B_total columns -> device slab `slot` (impala_ingest_shard)."""
        self._copy_to_slab(slot, "impala_ingest_shard", C.c_void_p(host_address), self.T, B_total, self.O, self.A,
                           b0, self.B)

    def load_device_batch(self, batch: dict, slot: int = 0) -> None:
        """Convenience for kernel-only timing: put a batch in HBM and wait for it."""
        self.fill_host(batch, slot)
        self.ingest(slot)
        self.copy_stream.synchronize()

    # ------------------------------------------------------------------------ step
    def _enqueue_main(self, slot: int = 0) -> int:
        lib, hp, st = self.lib, self.hp, C.c_void_p(torch.cuda.current_stream().cuda_stream)
        launched = lib.impala_launch_count()
        d = self.d_views[slot]
        T, B, O, A = self.T, self.B, self.O, self.A
        p_pi = C.c_void_p(self.params.data_ptr())
        p_vf = C.c_void_p(self.params.data_ptr() + 4 * self.n_pi)
        # this rank's [gradient | scalars] goes to `comm` (final at N = 1, reduced in place by NCCL,
        # source of impala_peer_push); the fused push variant of the backward sends the gradient
        # straight to the peers and only the scalars pass through `comm`
        gbase = self.comm.data_ptr()
        g_pi = C.c_void_p(gbase)
        g_vf = C.c_void_p(gbase + 8 * self.n_pi)
        scal = C.c_void_p(gbase + 8 * self.n_total)
        obs = _ptr(d["obs"])
        _cabi.check(lib.impala_mlp_forward_pair(obs, p_pi, p_vf, _ptr(self.logits), _ptr(self.values),
                                                self.M_pi, self.M_vf, O, self.H_pi, self.H_v, A, st),
                    "impala_mlp_forward_pair")
        _cabi.check(lib.impala_vtrace_loss(
            _ptr(self.logits), _ptr(d["beh_logits"]), _ptr(d["actions"]),
            _ptr(d["rewards"]), _ptr(d["done"]), _ptr(d["lens"]), _ptr(self.values),
            _ptr(self.vs), _ptr(self.pg_adv), _ptr(self.dlogits), _ptr(self.dv), scal,
            _ptr(self.ws_vt), self.ws_vt_bytes, T, B, A,
            float(hp.gamma), float(hp.rho_bar), float(hp.c_bar), float(hp.v_loss_c),
            float(hp.policy_loss_c), float(hp.entropy_c), float(self.inv_batch), self.mode, st),
            "impala_vtrace_loss")
        pr = self.peer
        if pr and pr["fused"]:
            _cabi.check(lib.impala_mlp_backward_pair_push(
                obs, p_pi, p_vf, _ptr(self.dlogits), _ptr(self.dv), _ptr(self.ws_pi), self.ws_pi_bytes,
                _ptr(self.ws_vf), self.ws_vf_bytes, self.M_pi, self.M_vf, O, self.H_pi, self.H_v, A, scal, 4,
                _ptr(pr["gather_ptrs"]), _ptr(pr["seq"]), pr["slot"], pr["buf"], pr["rank"], self.world, st),
                "impala_mlp_backward_pair_push")
        else:
            _cabi.check(lib.impala_mlp_backward_pair(
                obs, p_pi, p_vf, _ptr(self.dlogits), _ptr(self.dv), g_pi, g_vf, _ptr(self.ws_pi), self.ws_pi_bytes,
                _ptr(self.ws_vf), self.ws_vf_bytes, self.M_pi, self.M_vf, O, self.H_pi, self.H_v, A, st),
                "impala_mlp_backward_pair")
            if pr:  # stand-alone producer: comm[0 : n_total + 8) -> every rank's gather buffer
                _cabi.check(lib.impala_peer_push(_ptr(self.comm), self.n_total + 8, _ptr(pr["gather_ptrs"]),
                                                 _ptr(pr["seq"]), pr["slot"], pr["buf"], pr["rank"], self.world, st),
                            "impala_peer_push")
        return int(lib.impala_launch_count() - launched)  # kernels actually launched / captured

    def _enqueue_opt(self) -> int:
        hp, st = self.hp, C.c_void_p(torch.cuda.current_stream().cuda_stream)
        if self.peer:
            pr = self.peer
            _cabi.check(self.lib.impala_gather_clip_adam(
                _ptr(self.params), _ptr(self.comm), C.c_void_p(pr["gather"]), _ptr(pr["seq"]),
                pr["slot"], pr["buf"], self.world, 4, _ptr(self.adam_m), _ptr(self.adam_v), _ptr(self.adam_step),
                self.n_pi, self.n_total, float(hp.max_norm), float(0.95 * hp.lr), 0.9, 0.999, 1e-8,
                _ptr(self.norms), _ptr(pr["err"]), pr["timeout_s"], st), "impala_gather_clip_adam")
            return 1
        _cabi.check(self.lib.impala_clip_adam(
            _ptr(self.params), _ptr(self.comm), _ptr(self.adam_m), _ptr(self.adam_v),
            _ptr(self.adam_step), self.n_pi, self.n_total, float(hp.max_norm),
            float(0.95 * hp.lr),  # LambdaLR(lambda e: 0.95): constant factor, learner.py:42
            0.9, 0.999, 1e-8, _ptr(self.norms), st), "impala_clip_adam")
        return 1

    def _capture(self, slot: int):
        # thread_local: other host threads of the learner process (weight publisher, evaluation) keep
        # making CUDA calls while this thread captures
        with torch.cuda.stream(self.stream):
            g1 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g1, stream=self.stream, capture_error_mode="thread_local"):
                self._main_launches = self._enqueue_main(slot)
                if self._one_graph():  # no library collective in between: the optimizer joins the graph
                    self._enqueue_opt()
            self._graph_main[slot] = g1
            if not self._one_graph() and self._graph_opt is None:
                g2 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g2, stream=self.stream, capture_error_mode="thread_local"):
                    self._enqueue_opt()
                self._graph_opt = g2

    def _one_graph(self) -> bool:
        """Single GPU, or the all-reduce is the push over peer memory (no library call in between)."""
        return self.world == 1 or self.peer is not None

    def loop_stream(self, on: bool = True) -> None:
        """Make `self.stream` the calling thread's current stream for the duration of an update loop, so
        that step / post_scalars do not pay a stream-context switch per call (about 5 us each - the
        learner loop is host-bound at small batches).  loop_stream(False) restores the default stream."""
        import threading

        torch.cuda.set_stream(self.stream if on else torch.cuda.default_stream(self.dev))
        self._loop_thread = threading.get_ident() if on else None

    def _on_stream(self):
        import threading

        if self._loop_thread is not None and self._loop_thread == threading.get_ident():
            return contextlib.nullcontext()
        return torch.cuda.stream(self.stream)

    def step(self, slot: int = 0) -> None:
        """One learner update on the batch in device slab `slot` (async on `self.stream`)."""
        with self._on_stream():
            self.stream.wait_event(self.slab_ready[slot])
            if self.use_graph and self.steps_done >= 1:
                if slot not in self._graph_main:
                    self._capture(slot)
                self._graph_main[slot].replay()
                n = self._main_launches
                fused_opt = self._one_graph()
            else:
                n = self._enqueue_main(slot)  # first step eager: fills the launch-config caches
                fused_opt = False
            self.slab_free[slot].record(self.stream)
            self._slab_used[slot] = True
            if self.world > 1 and not self.peer:
                import torch.distributed as dist

                dist.all_reduce(self.comm, op=dist.ReduceOp.SUM, group=self.pg)
            if fused_opt:
                n += 1
            elif self.use_graph and self._graph_opt is not None:
                self._graph_opt.replay()
                n += 1
            else:
                n += self._enqueue_opt()
        self.launches_per_step = n
        self.steps_done += 1

    def forward_backward_only(self) -> None:
        """Everything up to (not including) the collective and the optimizer - for tests."""
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(self.slab_ready[0])
            self._enqueue_main(0)

    def read_scalars(self) -> dict:
        """D2H of the step's logged numbers (learner.py:217-240); waits for the step."""
        return self.fetch_scalars(self.post_scalars())

    def post_scalars(self) -> int:
        """Enqueue the D2H of the current step's scalars; returns a ticket for fetch_scalars."""
        k = self._ticket % 4
        self._ticket += 1
        with self._on_stream():
            self.h_scalars[k, :4].copy_(self.comm[self.n_total:self.n_total + 4], non_blocking=True)
            self.h_scalars[k, 4:6].copy_(self.norms, non_blocking=True)
            if self.peer:
                self.h_scalars[k, 6:7].copy_(self.peer["err"].to(torch.float64), non_blocking=True)
            self._scalar_events[k].record(self.stream)
        return k

    def fetch_scalars(self, ticket: int) -> dict:
        self._scalar_events[ticket].synchronize()
        s = self.h_scalars[ticket].tolist()
        if self.peer and s[6] != 0.0:
            raise _cabi.ImpalaCudaError(
                f"data-parallel learner: a peer rank did not deliver its gradient within {self.peer['timeout_s']:.0f} s "
                "(IMPALA_PEER_TIMEOUT_S); parameters were left untouched on this rank")
        hp = self.hp
        out = dict(zip(SCALAR_NAMES, s[:4]))
        out["total_loss"] = (hp.v_loss_c * out["value_fn_loss"] + hp.policy_loss_c * out["policy_loss"]
                             - hp.entropy_c * out["policy_entropy"])  # learner.py:154-159
        out["norm_policy"], out["norm_value"] = s[4], s[5]
        return out

    def synchronize(self) -> None:
        self.copy_stream.synchronize()
        self.stream.synchronize()
