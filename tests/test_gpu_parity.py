"""GPU parity: the sm_100a kernels (through the C ABI) against the float64 oracle.

Tolerance (BASELINE.json north_star): V-trace targets, pg advantages and the three loss
scalars within 1e-5 absolute of the reference in float32.  Gradients are compared
relative to their largest entry.  Inputs are the committed golden fixtures (outputs of
the real reference) plus seeded synthetic batches at sizes the oracle does in seconds.
"""
import numpy as np
import pytest
import torch

from conftest import PKEYS
from oracle import impala_oracle as orc
from torched_impala_b200 import synth
from torched_impala_b200.utils import default_hparams

pytestmark = pytest.mark.gpu

ATOL = 1e-5  # north_star tolerance


def scalar_tol(ref: float, u: int = 0) -> float:
    """1e-5, absolute up to magnitude 1 and relative beyond: the logged losses are sums over T*B
    float32 terms and reach O(10-100) (c1: value_fn_loss = 37.25, one float32 ulp = 3.8e-6), where
    an absolute 1e-5 sits at the rounding noise of ANY float32 evaluation order."""
    return ATOL * (1 + u) * max(1.0, abs(ref))


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device is visible")
    from torched_impala_b200 import ops as _ops

    return _ops


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def rel_err(got, want):
    scale = max(1e-30, float(np.abs(want).max()))
    return float(np.abs(got - want).max()) / scale


MLP_SHAPES = [
    # (M, O, H, N2)
    (21 * 8, 4, 32, 2), (21 * 8, 4, 32, 1), (1000, 7, 40, 3), (1000, 7, 24, 1),
    (20 * 64 + 5, 24, 256, 4), (21 * 64, 24, 256, 1), (333, 64, 512, 4), (333, 64, 512, 1),
    (97, 32, 128, 16), (64, 8, 100, 5), (4097, 24, 256, 4), (86016, 24, 256, 1), (700, 28, 96, 3),
    # wide tensor-core kernels (mlp_tcw.cu): O <= 64, H a multiple of 128, several tiles and passes per CTA
    (60001, 64, 512, 4), (60001, 64, 512, 1), (1000, 40, 384, 3), (130, 24, 512, 1), (257, 32, 128, 2),
    (5, 64, 512, 4), (129, 4, 512, 2),
]


@pytest.mark.parametrize("tensor_cores", ["1", "0"])
@pytest.mark.parametrize("M,O,H,N2", MLP_SHAPES)
def test_mlp_forward(ops, monkeypatch, M, O, H, N2, tensor_cores):
    """Both forward paths: tcgen05 3xTF32 (default where the layer is GEMM-shaped) and FP32 FFMA."""
    monkeypatch.setenv("IMPALA_MLP_TC", tensor_cores)
    rng = np.random.default_rng(M + O + H + N2)
    p = synth.init_params(M, O, N2, H)["policy"]
    x = rng.standard_normal((M, O), dtype=np.float32)
    want, _ = orc.mlp_forward(x.astype(np.float64), *[p[k].astype(np.float64) for k in PKEYS])
    got = ops.mlp_forward(dev(x), ops.pack_params(p), O, H, N2).cpu().numpy()
    assert got.shape == (M, N2)
    assert np.abs(got - want).max() < ATOL


@pytest.mark.parametrize("tensor_cores", ["1", "0"])
@pytest.mark.parametrize("M,O,H,N2", MLP_SHAPES + [(96, 4, 128, 1), (4100, 8, 256, 3), (2500, 28, 128, 4)])
def test_mlp_backward(ops, monkeypatch, M, O, H, N2, tensor_cores):
    """Both backward paths (tcgen05 3xTF32 for H in {128,256}, O%4==0, O<=28; FP32 FFMA otherwise).

    A ReLU unit whose pre-activation is within rounding of 0 may be switched differently than in
    float64; that moves one entry by one row's contribution, hence the tolerance term below."""
    monkeypatch.setenv("IMPALA_MLP_TC", tensor_cores)
    rng = np.random.default_rng(7 * M + O + H + N2)
    p = synth.init_params(M + 1, O, N2, H)["policy"]
    x = rng.standard_normal((M, O), dtype=np.float32)
    dout = (rng.standard_normal((M, N2), dtype=np.float32) / M).astype(np.float32)
    p64 = [p[k].astype(np.float64) for k in PKEYS]
    _, pre = orc.mlp_forward(x.astype(np.float64), *p64)
    want = orc.mlp_backward(x.astype(np.float64), pre, p64[2], dout.astype(np.float64))
    flat = ops.mlp_backward(dev(x), ops.pack_params(p), dev(dout), O, H, N2)
    got = ops.unpack_grad(flat, O, H, N2)
    one_row = float(np.abs(dout).max() * np.abs(p[PKEYS[2]]).max() * max(1.0, np.abs(x).max()))
    for k, w in zip(PKEYS, want):
        assert got[k].shape == w.shape
        tol = 2e-5 * np.abs(w).max() + (3 * one_row if k in PKEYS[:2] else 0.0)
        assert np.abs(got[k] - w).max() < tol, (k, rel_err(got[k], w))
    # pad entries of the parameter block must be exactly zero (they enter the clip norm)
    total = float(flat.abs().sum().cpu())
    real = sum(np.abs(g).sum() for g in got.values())
    assert abs(total - real) <= 1e-12 * max(1.0, real)


PAIR_SHAPES = [
    # (T, B, O, H_pi, H_vf, A): M_pi = T*B, M_vf = (T+1)*B
    (20, 64, 24, 256, 256, 4), (20, 1024, 24, 256, 256, 4), (5, 7, 8, 128, 256, 2), (3, 50, 28, 256, 128, 3),
    (20, 4096, 24, 256, 256, 4), (20, 8, 4, 32, 32, 2), (9, 33, 64, 512, 512, 4),
]


@pytest.mark.parametrize("T,B,O,H_pi,H_vf,A", PAIR_SHAPES)
def test_mlp_pair_matches_single_calls(ops, T, B, O, H_pi, H_vf, A):
    """impala_mlp_forward_pair / impala_mlp_backward_pair (both networks in one launch where the
    tensor-core path covers them, two launches otherwise) against the per-network entry points:
    the forward bit for bit, the backward to float64 rounding (only the number of float32 partial
    rows that are summed differs) - and so transitively against the oracle."""
    rng = np.random.default_rng(T * B + O)
    M_pi, M_vf = T * B, (T + 1) * B
    pp = ops.pack_params(synth.init_params(1, O, A, H_pi)["policy"])
    pv = ops.pack_params(synth.init_params(2, O, 1, H_vf)["policy"])
    x = dev(rng.standard_normal((M_vf, O), dtype=np.float32))
    dlog = dev((rng.standard_normal((M_pi, A), dtype=np.float32) / M_pi).astype(np.float32))
    dv = dev((rng.standard_normal((M_vf,), dtype=np.float32) / M_vf).astype(np.float32))
    logits, values = ops.mlp_forward_pair(x, pp, pv, M_pi, M_vf, O, H_pi, H_vf, A)
    assert torch.equal(logits, ops.mlp_forward(x[:M_pi], pp, O, H_pi, A))
    assert torch.equal(values, ops.mlp_forward(x, pv, O, H_vf, 1).reshape(-1))
    for rep in range(2):  # twice: the grid barrier re-arms itself
        g_pi, g_vf = ops.mlp_backward_pair(x, pp, pv, dlog, dv, O, H_pi, H_vf, A)
        for got, want in ((g_pi, ops.mlp_backward(x[:M_pi], pp, dlog, O, H_pi, A)),
                          (g_vf, ops.mlp_backward(x, pv, dv.reshape(-1, 1), O, H_vf, 1))):
            scale = float(want.abs().max())
            assert float((got - want).abs().max()) <= 5e-6 * scale + 1e-12, rep


def _oracle_forward(g, u):
    lrn = orc.BatchedLearner(g.init_params() if u == 0 else g.params_after(u - 1), g.hp)
    return lrn.forward_backward(g.batch(u))


def test_vtrace_matches_golden(ops, golden):
    """C-ABI impala_vtrace vs `vt` / `pg_adv` of the real reference (learner.py:127-135)."""
    for u in range(golden.updates):
        b = golden.batch(u)
        out = _oracle_forward(golden, u)
        hp = golden.hp
        vs, pg = ops.vtrace(dev(out["logits"], torch.float32), dev(b["beh_logits"]),
                            dev(b["actions"]), dev(b["rewards"]), dev(b["done"]), dev(b["lens"]),
                            dev(out["v"], torch.float32), hp.gamma, hp.rho_bar, hp.c_bar)
        assert np.abs(vs.cpu().numpy() - golden.z[f"u{u}_vs"]).max() < ATOL
        assert np.abs(pg.cpu().numpy() - golden.z[f"u{u}_pg_adv"]).max() < ATOL


def test_vtrace_loss_matches_golden(ops, golden):
    for u in range(golden.updates):
        b = golden.batch(u)
        out = _oracle_forward(golden, u)
        hp = golden.hp
        res = ops.vtrace_loss(dev(out["logits"], torch.float32), dev(b["beh_logits"]),
                              dev(b["actions"]), dev(b["rewards"]), dev(b["done"]), dev(b["lens"]),
                              dev(out["v"], torch.float32), hp, 1.0 / hp.batch_size)
        sc = res["scalars"].cpu().numpy()
        ref = golden.scalars(u)
        for i, k in enumerate(("value_fn_loss", "policy_loss", "policy_entropy", "batch_mean_reward")):
            assert abs(sc[i] - ref[k]) < ATOL, (k, sc[i], ref[k])
        assert np.abs(res["vs"].cpu().numpy() - golden.z[f"u{u}_vs"]).max() < ATOL
        assert np.abs(res["pg_adv"].cpu().numpy() - golden.z[f"u{u}_pg_adv"]).max() < ATOL
        assert rel_err(res["dlogits"].cpu().numpy(), out["dlogits"]) < 2e-5
        assert rel_err(res["dv"].cpu().numpy(), out["dv"]) < 2e-5


@pytest.mark.parametrize("T,B,A,ragged,mode", [
    (20, 256, 2, False, "reference"), (33, 19, 3, True, "reference"), (64, 8, 4, True, "reference"),
    (100, 512, 4, False, "reference"), (128, 24, 4, True, "reference"), (129, 9, 4, True, "reference"),
    (300, 16, 6, True, "reference"), (1000, 8, 2, True, "reference"), (40, 40, 16, True, "reference"),
    (20, 64, 4, True, "paper"), (256, 8, 4, False, "paper"),
])
def test_vtrace_loss_synthetic(ops, T, B, A, ragged, mode):
    """Ragged / long / odd shapes (chunked unrolls, partial CTAs) against the batched oracle."""
    hp = default_hparams(batch_size=B, rho_bar=0.9, c_bar=0.8, gamma=0.97)
    b = synth.make_batch(T * 7 + B, T, B, 3, A, ragged=ragged)
    rng = np.random.default_rng(T + B + A)
    logits = rng.standard_normal((T, B, A), dtype=np.float32)
    v = rng.standard_normal((T + 1, B), dtype=np.float32)
    vs, pg, _ = orc.vtrace(v, logits, b["beh_logits"], b["actions"], b["rewards"], b["done"],
                           b["lens"], hp.gamma, hp.rho_bar, hp.c_bar, mode)
    ref = orc.losses(v.astype(np.float64), vs, logits, b["actions"], pg, b["lens"], hp.v_loss_c,
                     hp.policy_loss_c, hp.entropy_c, B)
    res = ops.vtrace_loss(dev(logits), dev(b["beh_logits"]), dev(b["actions"]), dev(b["rewards"]),
                          dev(b["done"]), dev(b["lens"]), dev(v), hp, 1.0 / B, mode=mode)
    assert np.abs(res["vs"].cpu().numpy() - vs).max() < ATOL * max(1.0, np.abs(vs).max() / 10)
    assert np.abs(res["pg_adv"].cpu().numpy() - pg).max() < ATOL * max(1.0, np.abs(pg).max() / 10)
    sc = res["scalars"].cpu().numpy()
    for i, k in enumerate(("value_fn_loss", "policy_loss", "policy_entropy")):
        assert abs(sc[i] - ref[k]) < ATOL * max(1.0, abs(ref[k]) / 10), (k, sc[i], ref[k])
    assert rel_err(res["dlogits"].cpu().numpy(), ref["dlogits"]) < 2e-5
    assert rel_err(res["dv"].cpu().numpy(), ref["dv"]) < 2e-5
    vs2, pg2 = ops.vtrace(dev(logits), dev(b["beh_logits"]), dev(b["actions"]), dev(b["rewards"]),
                          dev(b["done"]), dev(b["lens"]), dev(v), hp.gamma, hp.rho_bar, hp.c_bar,
                          mode=mode)
    assert torch.equal(vs2, res["vs"]) and torch.equal(pg2, res["pg_adv"])


def test_vtrace_quirk_is_reproduced(ops):
    """Fails if someone 'fixes' learner.py:126/130: reference mode must differ from paper mode."""
    T, B, A = 20, 32, 4
    b = synth.make_batch(5, T, B, 3, A)
    rng = np.random.default_rng(0)
    logits = rng.standard_normal((T, B, A), dtype=np.float32)
    v = rng.standard_normal((T + 1, B), dtype=np.float32)
    args = (dev(logits), dev(b["beh_logits"]), dev(b["actions"]), dev(b["rewards"]), dev(b["done"]),
            dev(b["lens"]), dev(v), 0.99, 1.0, 1.0)
    vs_ref, _ = ops.vtrace(*args, mode="reference")
    vs_pap, _ = ops.vtrace(*args, mode="paper")
    assert (vs_ref - vs_pap).abs().max().item() > 1e-2


@pytest.mark.parametrize("n_pi,n_vf,max_norm", [(419 - 97, 97, 10.0), (7456, 6688, 0.05), (70000, 66000, 1.0)])
def test_clip_adam(ops, n_pi, n_vf, max_norm):
    rng = np.random.default_rng(n_pi)
    n = n_pi + n_vf
    p0 = rng.standard_normal(n).astype(np.float32)
    params = dev(p0)
    m = torch.zeros(n, device="cuda")
    v = torch.zeros(n, device="cuda")
    step = torch.zeros(3, dtype=torch.int64, device="cuda")  # step, beta1^t, beta2^t
    hp = default_hparams(max_norm=max_norm, lr=1e-3)
    ref_p = [p0[:n_pi].astype(np.float64), p0[n_pi:].astype(np.float64)]
    adam = orc.Adam(ref_p, hp.lr)
    for it in range(3):
        g = rng.standard_normal(n) * (0.01 if it else 1.0)
        norms = ops.clip_adam(params, dev(g), m, v, step, n_pi, max_norm, 0.95 * hp.lr)
        c0, n0 = orc.clip_coef([g[:n_pi]], max_norm)
        c1, n1 = orc.clip_coef([g[n_pi:]], max_norm)
        adam.step(ref_p, [g[:n_pi] * c0, g[n_pi:] * c1])
        nn = norms.cpu().numpy()
        assert abs(nn[0] - n0) < 1e-9 * max(1, n0) and abs(nn[1] - n1) < 1e-9 * max(1, n1)
        got = params.cpu().numpy()
        assert np.abs(got - np.concatenate(ref_p)).max() < 3e-6
    assert int(step[0].item()) == 3


def _engine_for(g, use_graph):
    from torched_impala_b200.engine import LearnerEngine

    c = g.case
    eng = LearnerEngine(c["T"], c["B"], c["O"], c["A"], c["H_pi"], c["H_v"], g.hp,
                        use_graph=use_graph)
    eng.load_state(g.init_params())
    return eng


@pytest.mark.parametrize("use_graph", [False, True])
def test_engine_updates_match_reference(golden, use_graph):
    """Whole learner steps (ingest -> ... -> Adam) against scalars / params of learner.py."""
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device is visible")
    eng = _engine_for(golden, use_graph)
    for u in range(golden.updates):
        eng.fill_host(golden.batch(u), u % 2)
        eng.ingest(u % 2)
        eng.step(u % 2)
        sc = eng.read_scalars()
        ref = golden.scalars(u)
        for k in ("value_fn_loss", "policy_loss", "policy_entropy", "total_loss", "batch_mean_reward"):
            assert abs(sc[k] - ref[k]) < scalar_tol(ref[k], u), (u, k, sc[k], ref[k])
        assert np.abs(eng.vs.cpu().numpy() - golden.z[f"u{u}_vs"]).max() < ATOL * (1 + u)
        assert np.abs(eng.pg_adv.cpu().numpy() - golden.z[f"u{u}_pg_adv"]).max() < ATOL * (1 + u)
        if u == 0:
            got, want = eng.grads(), golden.raw_grads(0)
            for grp in want:
                for k in PKEYS:
                    assert rel_err(golden.pick(grp, k, got[grp][k]), want[grp][k]) < 3e-5, (grp, k)
        st, want = eng.state(), golden.params_after(u)
        for grp in want:
            for k in PKEYS:
                d = np.abs(golden.pick(grp, k, st[grp][k].numpy()) - want[grp][k]).max()
                assert d < 2e-5 * (1 + u), (u, grp, k, d)


def test_full_size_properties():
    """c4 shape (T=20, B=4096, O=24, H=256): size-independent checks, no oracle pass needed.

    (1) padding neutrality: the same trajectories embedded in a longer unroll give the same
    scalars and gradients; (2) shard additivity: two half-batches with inv_batch of the full
    batch sum to the full-batch gradient and scalars (what the all-reduce relies on)."""
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device is visible")
    from torched_impala_b200.engine import LearnerEngine

    T, B, O, A, H = 20, 4096, 24, 4, 256
    hp = default_hparams(batch_size=B)
    params = synth.init_params(1, O, A, H)
    batch = synth.make_batch(2, T, B, O, A, ragged=True)

    def run(T_, b, Bl, gb):
        e = LearnerEngine(T_, Bl, O, A, H, H, hp, global_batch=gb, use_graph=False)
        e.load_state(params)
        e.load_device_batch(b)
        e.forward_backward_only()
        e.synchronize()
        return e.comm.cpu().numpy().copy()

    full = run(T, batch, B, B)
    wide = {k: (v if k == "lens" else np.concatenate([v, np.zeros((5,) + v.shape[1:], v.dtype)], 0))
            for k, v in batch.items()}
    padded = run(T + 5, wide, B, B)
    scale = np.abs(full).max()
    assert np.abs(full - padded).max() < 1e-5 * scale
    halves = sum(run(T, synth.shard_batch(batch, r, 2), B // 2, B) for r in range(2))
    assert np.abs(full - halves).max() < 1e-5 * scale


def test_loss_helper_functions_match_reference_formulas():
    """The four module-level helpers of learner.py:298-321 (values and gradients), float64 torch on
    the CPU as the reference of the formulas."""
    import torch.nn.functional as F

    from torched_impala_b200 import learner as L

    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device is visible")
    torch.manual_seed(0)
    Lr, A = 37, 5
    z = torch.randn(Lr, A, dtype=torch.float64, requires_grad=True)
    a = torch.randint(0, A, (Lr, 1))
    adv = torch.randn(Lr, dtype=torch.float64)
    lsm = F.log_softmax(z, -1)
    ref = dict(alp=lsm.gather(-1, a), base=0.5 * (adv ** 2).sum(), ent=(lsm.exp() * lsm).sum(),
               pg=(-lsm.gather(-1, a).view(-1) * adv).sum())
    g_ref = torch.autograd.grad(ref["ent"] * 0.3 + ref["pg"] * 1.7 + ref["alp"].sum() * 0.5, z)[0]
    zc = z.detach().cuda().requires_grad_(True)
    ac, advc = a.cuda(), adv.cuda().requires_grad_(True)
    got = dict(alp=L.action_log_probs(zc, ac), base=L.compute_baseline_loss(advc),
               ent=L.compute_entropy_loss(zc), pg=L.compute_policy_gradient_loss(zc, ac, advc))
    assert got["alp"].shape == a.shape and got["alp"].dtype == torch.float64
    for k in ref:
        assert (got[k].detach().cpu() - ref[k].detach()).abs().max() < 1e-5, k
    (got["ent"] * 0.3 + got["pg"] * 1.7 + got["alp"].sum() * 0.5 + got["base"]).backward()
    assert (zc.grad.cpu() - g_ref).abs().max() < 1e-5
    assert (advc.grad.cpu() - adv).abs().max() < 1e-5  # d(0.5 sum adv^2) = adv; pg loss detaches adv
