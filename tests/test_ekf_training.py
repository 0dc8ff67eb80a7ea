"""Training the Kalman-filter models through the EKF kernels: ``training.FusedEKFLoop`` (mmf_ekf_loop_train_fwd records
the tape, mmf_ekf_loop_bwd walks the adjoint backwards in time) and the dispatch that selects it.

CPU: the adjoint, restated in float64 torch the way the kernel computes it, against torch.autograd through the oracle's
generic recursion (whose dynamics Jacobian is taken at a detached state); the structural dispatch checks.
GPU: the tape forward against ``ops.ekf_loop`` bit for bit, the kernel's gradients against a float64 recursion fed the
same tape, whole models against the generic fp32 path and the float64 oracle port, chaining across calls, determinism,
launch counts and ``train_e2e``."""
import numpy as np
import pytest
import torch

from oracle import crossmodal_port as port  # installs the oracle shims on sys.path

import torchfilter  # noqa: E402  (the oracle shim)
from multimodalfilter_b200 import fused, training  # noqa: E402
from multimodalfilter_b200.crossmodal import models as M  # noqa: E402
from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories  # noqa: E402

DEV = "cuda:0"
f64 = torch.float64


# ---- the adjoint, restated ----------------------------------------------------------------------------------------
def ekf_adjoint(A, pred, covs, cov0, z, R, Q, d_means, d_covs):
    """The reverse mode of the EKF recursion as k_ekf_loop_bwd computes it, batched over the leading axis N:
    A, covs, R, d_covs (T,N,sd,sd); pred, z, d_means (T,N,sd); cov0 (N,sd,sd); Q = q q^T (sd,sd).  Reverse time,
    recompute Pp, S^-1, K from the stored posterior of step t-1 and the tape.  -> d_mean0, d_cov0, d_z, d_r."""
    T, N, sd = z.shape
    tr = lambda X: X.transpose(-1, -2)  # noqa: E731
    eye = torch.eye(sd, dtype=z.dtype)
    mb, Pb = torch.zeros(N, sd, dtype=z.dtype), torch.zeros(N, sd, sd, dtype=z.dtype)
    d_z, d_r = torch.zeros_like(z), torch.zeros_like(R)
    for t in reversed(range(T)):
        P = covs[t - 1] if t > 0 else cov0
        Pp = A[t] @ P @ tr(A[t]) + Q
        Si = torch.inverse(Pp + R[t] @ tr(R[t]))
        K = Pp @ Si
        r = z[t] - pred[t]
        mb = mb + d_means[t]
        if d_covs is not None:
            Pb = Pb + d_covs[t]
        d_z[t] = (tr(K) @ mb[..., None])[..., 0]
        mbp = mb - d_z[t]
        Kb = mb[..., None] * r[..., None, :] - Pb @ tr(Pp)
        Sb = -tr(Si) @ tr(Pp) @ Kb @ tr(Si)
        Ppb = tr(eye - K) @ Pb + Kb @ tr(Si) + Sb
        d_r[t] = (Sb + tr(Sb)) @ R[t]
        Pb = tr(A[t]) @ Ppb @ A[t]
        mb = (tr(A[t]) @ mbp[..., None])[..., 0]
    return mb, Pb, d_z, d_r


class _ToyDynamics(torchfilter.base.DynamicsModel):
    """x + 0.4 tanh(W x + B u + b): nonlinear, so A varies along the trajectory."""

    def __init__(self, sd, cd, g):
        super().__init__(state_dim=sd)
        self.W = torch.randn(sd, sd, generator=g, dtype=f64)
        self.B = torch.randn(sd, cd, generator=g, dtype=f64)
        self.b = torch.randn(sd, generator=g, dtype=f64)
        self.q = torch.tril(0.1 * torch.randn(sd, sd, generator=g, dtype=f64)) + 0.3 * torch.eye(sd, dtype=f64)

    def forward(self, *, initial_states, controls):
        x = initial_states
        y = x + 0.4 * torch.tanh(x @ self.W.T + controls @ self.B.T + self.b)
        return y, self.q[None].expand(x.shape[0], *self.q.shape)


class _GivenSensor(torchfilter.base.VirtualSensorModel):
    def forward(self, *, observations):
        return observations["z"], observations["r"]


@pytest.mark.parametrize("sd", [1, 2, 3, 4])
@pytest.mark.parametrize("T", [1, 17])
@pytest.mark.parametrize("with_d_covs", [True, False])
def test_adjoint_restatement_equals_autograd_through_the_generic_recursion(sd, T, with_d_covs):
    g = torch.Generator().manual_seed(100 * sd + T)
    N, cd = 5, 2
    dyn = _ToyDynamics(sd, cd, g)
    ekf = torchfilter.filters.VirtualSensorExtendedKalmanFilter(dynamics_model=dyn, virtual_sensor_model=_GivenSensor(state_dim=sd))
    mean0 = torch.randn(N, sd, generator=g, dtype=f64).requires_grad_(True)
    L0 = torch.randn(N, sd, sd, generator=g, dtype=f64)
    cov0 = (L0 @ L0.transpose(-1, -2) * 0.1 + 0.2 * torch.eye(sd, dtype=f64)).requires_grad_(True)
    z = torch.randn(T, N, sd, generator=g, dtype=f64).requires_grad_(True)
    R = (torch.tril(0.2 * torch.randn(T, N, sd, sd, generator=g, dtype=f64)) + 0.5 * torch.eye(sd, dtype=f64)).requires_grad_(True)
    u = torch.randn(T, N, cd, generator=g, dtype=f64)
    d_means = torch.randn(T, N, sd, generator=g, dtype=f64)
    d_covs = torch.randn(T, N, sd, sd, generator=g, dtype=f64) if with_d_covs else None

    ekf.initialize_beliefs(mean=mean0, covariance=cov0)
    means, covs, preds, jacs = [], [], [], []
    for t in range(T):
        preds.append(dyn(initial_states=ekf.belief_mean, controls=u[t])[0].detach())
        jacs.append(dyn.jacobian(initial_states=ekf.belief_mean, controls=u[t]).detach())
        ekf(observations={"z": z[t], "r": R[t]}, controls=u[t])
        means.append(ekf.belief_mean)
        covs.append(ekf.belief_covariance)
    means, covs = torch.stack(means), torch.stack(covs)
    loss = (means * d_means).sum() + ((covs * d_covs).sum() if with_d_covs else 0.0)
    want = torch.autograd.grad(loss, (mean0, cov0, z, R))

    got = ekf_adjoint(torch.stack(jacs), torch.stack(preds), covs.detach(), cov0.detach(), z.detach(), R.detach(),
                      dyn.q @ dyn.q.T, d_means, d_covs)
    for name, a, b in zip(("d_mean0", "d_cov0", "d_z", "d_r_tril"), got, want):
        rel = float((a - b).norm() / b.norm().clamp_min(1e-300))
        assert rel <= 1e-10, f"{name}: relative error {rel:.3e}"


# ---- dispatch (structural checks: no device needed) ---------------------------------------------------------------
def _frozen(model):
    filters = list(model.filter_models) if hasattr(model, "filter_models") else [model]
    for f in filters:
        for p in f.dynamics_model.parameters():
            p.requires_grad_(False)
    return filters


def _plan(filters):
    return fused.EKFPlan.build(filters)


@pytest.mark.parametrize("name", ["DoorKalmanFilter", "DoorCrossmodalKalmanFilter", "PushUnimodalKalmanFilter",
                                  "DoorMeasurementCrossmodalKalmanFilter"])
def test_dispatch_structure(name):
    model = getattr(M, name)()
    filters = _frozen(model)
    assert training.ekf_train_structure_ok(model, filters, _plan(filters)), "frozen dynamics must select the fused path"

    model.fused_train = False
    assert not training.ekf_train_structure_ok(model, filters, _plan(filters))
    assert all(not f.fused_train for f in filters)  # the member filters follow the switch
    model.fused_train = True

    p = next(filters[0].dynamics_model.parameters())
    p.requires_grad_(True)
    assert not training.ekf_train_structure_ok(model, filters, _plan(filters)), "trainable dynamics stay generic"
    p.requires_grad_(False)

    handle = filters[-1].virtual_sensor_model.register_forward_hook(lambda *a: None)
    assert not training.ekf_train_structure_ok(model, filters, _plan(filters)), "a hook keeps the generic path"
    handle.remove()
    assert training.ekf_train_structure_ok(model, filters, _plan(filters))

    class Odd(torch.nn.Module):
        state_dim = filters[0].state_dim

    odd = [type("F", (), {"dynamics_model": Odd()})()]
    assert _plan(odd) is None and not training.ekf_train_structure_ok(model, odd, _plan(odd)), \
        "an unrecognised dynamics module keeps the generic path"


def test_dispatch_needs_grad_and_cuda_fp32():
    model = M.DoorKalmanFilter()
    filters = _frozen(model)
    plan = _plan(filters)
    ctrl = torch.zeros(4, 7)
    obs = {"image": torch.zeros(4, 32, 32)}
    beliefs = (torch.zeros(4, 3), torch.zeros(4, 3, 3))
    assert not training.fused_ekf_train_applicable(model, filters, plan, ctrl, obs, beliefs), "CPU tensors stay generic"
    with torch.no_grad():
        assert not training.fused_ekf_train_applicable(model, filters, plan, ctrl, obs, beliefs)


# ---- GPU ----------------------------------------------------------------------------------------------------------
def _structs(F, sd, seed):
    """F recognised dynamics (sd 1 ... 4: the door model's layout with its state width changed)."""
    plans = []
    for f in range(F):
        noise = ("tril", [0.05, 0.01, 0.01, 0.02][:sd], 1.0)
        cls = type(f"Dyn{sd}", (M._Dynamics,), {"_STATE_DIM": sd, "_NOISE": noise})
        dyn = fill_parameters(cls(), seed=seed + f).to(DEV)
        for p in dyn.parameters():
            p.requires_grad_(False)
        plans.append(type("H", (), {"dynamics_model": dyn})())
    plan = fused.EKFPlan.build(plans)
    assert plan is not None
    return plan


def _inputs(F, T, N, sd, seed):
    g = torch.Generator().manual_seed(seed)
    mean0 = torch.randn(F, N, sd, generator=g)
    cov0 = (0.1 * torch.eye(sd)).expand(F, N, sd, sd).contiguous()
    z = torch.randn(F, T, N, sd, generator=g)
    R = torch.tril(0.05 * torch.randn(F, T, N, sd, sd, generator=g))
    R = R + torch.diag_embed(0.1 + torch.rand(F, T, N, sd, generator=g))  # diagonal >= 0.1: well conditioned
    u = torch.randn(T, N, 7, generator=g)
    return [x.to(DEV).contiguous() for x in (mean0, cov0, u, z, R)]


@pytest.mark.gpu
@pytest.mark.parametrize("F", [1, 2, 3, 4])
@pytest.mark.parametrize("sd", [1, 2, 3, 4])
def test_tape_forward_equals_ekf_loop_bit_for_bit(F, sd):
    plan = _structs(F, sd, seed=10)
    for N in (1, 33, 256):
        for T in (1, 16):
            mean0, cov0, u, z, R = _inputs(F, T, N, sd, seed=N + T)
            means, covs = plan.loop(mean0, cov0, u, z, R)
            tm, tc, pred, jac = plan.loop_train(mean0, cov0, u, z, R)
            assert torch.equal(means, tm) and torch.equal(covs, tc), (N, T)
            # the tape is the forward's own A and mu-: step 0 agrees with the standalone Jacobian kernel
            for f in range(F):
                p0, a0 = plan.jacobian(f, mean0[f], u[0])
                assert torch.equal(pred[f, 0], p0) and torch.equal(jac[f, 0], a0)


def _tape_recursion_grads(plan, mean0, cov0, u, z, R, d_means, d_covs):
    """float64 torch recursion fed A / mu- from the tape (mu-_t = pred_t + A_t (mu_{t-1} - mu_{t-1}.detach()): the value
    of the tape, the derivative A), differentiated by autograd."""
    means, covs, pred, jac = plan.loop_train(mean0, cov0, u, z, R)
    F, T, N, sd = z.shape
    # q_tril holds the sd x sd factor row-major in its first sd * sd entries (fused._DynamicsSpec.q)
    Q = torch.stack([torch.tensor(list(s.q_tril)[:sd * sd], dtype=f64).reshape(sd, sd) for s in plan.structs])
    Q = (Q @ Q.transpose(-1, -2)).to(DEV)[:, None]
    m0, P0, zz, RR = (x.double().requires_grad_(True) for x in (mean0, cov0, z, R))
    A, pr = jac.double(), pred.double()
    mu, P, outs_m, outs_P = m0, P0, [], []
    eye = torch.eye(sd, dtype=f64, device=DEV)
    for t in range(T):
        mp = pr[:, t] + (A[:, t] @ (mu - mu.detach())[..., None])[..., 0]
        Pp = A[:, t] @ P @ A[:, t].transpose(-1, -2) + Q
        S = Pp + RR[:, t] @ RR[:, t].transpose(-1, -2)
        K = Pp @ torch.inverse(S)
        mu = mp + (K @ (zz[:, t] - mp)[..., None])[..., 0]
        P = (eye - K) @ Pp
        outs_m.append(mu)
        outs_P.append(P)
    loss = (torch.stack(outs_m, 1) * d_means.double()).sum()
    if d_covs is not None:
        loss = loss + (torch.stack(outs_P, 1) * d_covs.double()).sum()
    return (means, covs, pred, jac), torch.autograd.grad(loss, (m0, P0, zz, RR))


@pytest.mark.gpu
@pytest.mark.parametrize("sd", [1, 2, 3, 4])
@pytest.mark.parametrize("with_d_covs", [True, False])
def test_backward_kernel_matches_float64_given_the_tape(sd, with_d_covs):
    from multimodalfilter_b200 import ops

    F, T, N = 2, 16, 33
    plan = _structs(F, sd, seed=20)
    mean0, cov0, u, z, R = _inputs(F, T, N, sd, seed=21)
    g = torch.Generator().manual_seed(22)
    d_means = torch.randn(F, T, N, sd, generator=g).to(DEV)
    d_covs = torch.randn(F, T, N, sd, sd, generator=g).to(DEV) if with_d_covs else None
    (means, covs, pred, jac), want = _tape_recursion_grads(plan, mean0, cov0, u, z, R, d_means, d_covs)
    got = ops.ekf_loop_bwd(plan.structs, cov0, z, R, covs, pred, jac, d_means, d_covs)
    worst = 0.0
    for name, a, b in zip(("d_mean0", "d_cov0", "d_z", "d_r_tril"), got, want):
        rel = float((a.double() - b).norm() / b.norm())
        worst = max(worst, rel)
        assert rel <= 1e-4, f"{name}: relative L2 {rel:.2e}"
    print(f"sd={sd} d_covs={'given' if with_d_covs else 'NULL'}: largest relative L2 error {worst:.2e}")


def _image_encoder(name):
    return "observation_image_layers" in name


def _model_case(name, know_blackout=False):
    def make(src):
        cls = getattr(src, name)
        return cls(know_image_blackout=True) if know_blackout else cls()

    return make


KF_CASES = [
    ("DoorKalmanFilter", 3, {}),
    ("DoorCrossmodalKalmanFilter", 3, {}),
    ("DoorCrossmodalKalmanFilter", 3, {"know_blackout": True}),
    ("DoorCrossmodalKalmanFilter", 3, {"disabled": True}),
    ("DoorUnimodalKalmanFilter", 3, {}),
    ("PushCrossmodalKalmanFilter", 2, {}),
    ("DoorMeasurementCrossmodalKalmanFilter", 3, {}),
]


def _run_model(model, states, obs, controls, dev, dtype, fused_train=None, freeze_images=True, disabled=False):
    model = model.to(dev, dtype).train()
    for p in model.dynamics_model.parameters() if hasattr(model, "dynamics_model") else []:
        p.requires_grad_(False)
    for f in getattr(model, "filter_models", []):
        for p in f.dynamics_model.parameters():
            p.requires_grad_(False)
    if freeze_images:
        for n, p in model.named_parameters():
            if _image_encoder(n):
                p.requires_grad_(False)
    if disabled:
        model._enabled_models = [False, True]
    if fused_train is not None:
        model.fused_train = fused_train
    sd = model.state_dim
    N = states.shape[1]
    cov = (torch.eye(sd, dtype=dtype) * 0.1)[None].expand(N, sd, sd).to(dev).contiguous()
    model.initialize_beliefs(mean=states[0].to(dev, dtype), covariance=cov)
    est = model.forward_loop(observations={k: v[1:].to(dev, dtype) for k, v in obs.items()},
                             controls=controls[1:].to(dev, dtype))
    loss = torch.mean((est - states[1:].to(dev, dtype)) ** 2)
    loss.backward()
    grads = {k: p.grad.detach().double().cpu() for k, p in model.named_parameters() if p.grad is not None}
    return float(loss), grads


@pytest.mark.gpu
@pytest.mark.parametrize("name,sd,opts", KF_CASES)
@pytest.mark.parametrize("freeze_images", [True, False])
def test_models_fused_vs_generic_vs_float64(name, sd, opts, freeze_images):
    from multimodalfilter_b200 import ops

    T, N = 16, 32
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=31, blackout_fraction=0.3 if opts.get("know_blackout") else 0)
    make = _model_case(name, opts.get("know_blackout", False))
    kw = dict(freeze_images=freeze_images, disabled=opts.get("disabled", False))
    ops.PROFILE.reset(enabled=True)
    l_fused, g_fused = _run_model(fill_parameters(make(M), seed=32), states, obs, controls, DEV, torch.float32, **kw)
    kernels = ops.PROFILE.collect()["kernels"]
    ops.PROFILE.reset()
    assert kernels.get("ekf_loop_train", {}).get("count") == 1 and kernels.get("ekf_loop_bwd", {}).get("count") == 1, kernels
    l_gen, g_gen = _run_model(fill_parameters(make(M), seed=32), states, obs, controls, DEV, torch.float32,
                              fused_train=False, **kw)
    l_ref, g_ref = _run_model(fill_parameters(make(port), seed=32), states, obs, controls, "cpu", f64, **kw)
    assert set(g_fused) == set(g_gen) == set(g_ref) and len(g_ref) > 0
    if freeze_images:
        assert abs(l_fused - l_ref) <= 2 * abs(l_gen - l_ref) + 1e-6 * abs(l_ref), (l_fused, l_gen, l_ref)
        for k in g_ref:
            scale = float(g_ref[k].norm()) or 1.0
            e_f = float((g_fused[k] - g_ref[k]).norm()) / scale
            e_g = float((g_gen[k] - g_ref[k]).norm()) / scale
            assert e_f <= 2 * e_g + 1e-6, f"{k}: fused {e_f:.2e} vs generic {e_g:.2e} (relative to float64)"
    else:
        assert abs(l_fused - l_gen) <= 1e-5 * abs(l_gen)
        big = max(float(g.norm()) for g in g_gen.values())
        for k in g_gen:
            a, b = g_fused[k].reshape(-1), g_gen[k].reshape(-1)
            rel = float((a - b).norm() / max(float(b.norm()), 1e-3 * big))
            cos = float(torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-30)) if float(b.norm()) > 1e-3 * big else 1.0
            assert rel <= 2e-2 and cos >= 0.999, f"{k}: relative L2 {rel:.2e}, cosine {cos:.5f}"


def _fresh(name, seed=41):
    m = fill_parameters(getattr(M, name)(), seed=seed).to(DEV).train()
    for f in getattr(m, "filter_models", [m]):
        for p in f.dynamics_model.parameters():
            p.requires_grad_(False)
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["DoorKalmanFilter", "DoorCrossmodalKalmanFilter", "DoorUnimodalKalmanFilter"])
def test_forward_steps_and_split_loops_chain_the_gradient(name):
    """T calls of forward against one forward_loop (the T = 1 path, chaining through mean0 / cov0), and two forward_loop
    calls of T steps against one of 2T."""
    from multimodalfilter_b200 import ops

    T, N, sd = 8, 16, 3
    states, obs, controls = synthetic_trajectories(2 * T + 1, N, sd, seed=42)
    o = {k: v[1:].to(DEV) for k, v in obs.items()}
    c, target = controls[1:].to(DEV), states[1:].to(DEV)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(DEV).contiguous()

    def run(mode):
        m = _fresh(name)
        m.initialize_beliefs(mean=states[0].to(DEV), covariance=cov)
        ops.PROFILE.reset(enabled=True)
        if mode == "loop":
            est = m.forward_loop(observations=o, controls=c)
        elif mode == "split":
            h = {k: v[:T] for k, v in o.items()}
            est = torch.cat([m.forward_loop(observations=h, controls=c[:T]),
                             m.forward_loop(observations={k: v[T:] for k, v in o.items()}, controls=c[T:])])
        else:
            est = torch.stack([m(observations={k: v[t] for k, v in o.items()}, controls=c[t]) for t in range(2 * T)])
        loss = torch.mean((est - target) ** 2)
        loss.backward()
        kernels = ops.PROFILE.collect()["kernels"]
        ops.PROFILE.reset()
        assert "ekf_loop_train" in kernels and "ekf_loop_bwd" in kernels and "ekf_loop" not in kernels, kernels
        return float(loss), {k: p.grad.double().cpu() for k, p in m.named_parameters() if p.grad is not None}

    l0, g0 = run("loop")
    for mode in ("split", "steps"):
        l1, g1 = run(mode)
        assert abs(l1 - l0) <= 1e-5 * abs(l0), (mode, l0, l1)
        assert set(g1) == set(g0)
        big = max(float(g.norm()) for g in g0.values())
        for k in g0:
            rel = float((g1[k] - g0[k]).norm() / max(float(g0[k].norm()), 1e-3 * big))
            assert rel <= 2e-3, f"{mode} {k}: relative L2 {rel:.2e}"


@pytest.mark.gpu
def test_measurement_initialize_carries_the_gradient_into_the_virtual_sensors():
    T, N, sd = 8, 16, 3
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=51)
    o = {k: v.to(DEV) for k, v in obs.items()}
    results = []
    for fused_train in (True, False):
        m = _fresh("DoorCrossmodalKalmanFilter", seed=52)
        m.fused_train = fused_train
        m.measurement_initialize_beliefs(observations={k: v[0] for k, v in o.items()})
        assert m.filter_models[0]._belief_mean.requires_grad
        est = m.forward_loop(observations={k: v[1:] for k, v in o.items()}, controls=controls[1:].to(DEV))
        loss = torch.mean((est - states[1:].to(DEV)) ** 2)
        loss.backward()
        results.append((float(loss), {k: p.grad.double().cpu() for k, p in m.named_parameters() if p.grad is not None}))
    (l0, g0), (l1, g1) = results
    assert abs(l0 - l1) <= 1e-5 * abs(l1) and set(g0) == set(g1)
    big = max(float(g.norm()) for g in g1.values())
    for k in g1:
        a, b = g0[k].reshape(-1), g1[k].reshape(-1)
        rel = float((a - b).norm() / max(float(b.norm()), 1e-3 * big))
        assert rel <= 2e-2, f"{k}: relative L2 {rel:.2e}"


@pytest.mark.gpu
def test_backward_is_bit_reproducible():
    T, N, sd = 16, 64, 3
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=61)
    runs = []
    for _ in range(2):
        m = _fresh("DoorCrossmodalKalmanFilter", seed=62)
        for n, p in m.named_parameters():
            if _image_encoder(n):  # cuDNN's convolution backward is outside this library's control
                p.requires_grad_(False)
        cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(DEV).contiguous()
        mean0 = states[0].to(DEV).requires_grad_(True)
        m.initialize_beliefs(mean=mean0, covariance=cov)
        est = m.forward_loop(observations={k: v[1:].to(DEV) for k, v in obs.items()}, controls=controls[1:].to(DEV))
        torch.mean((est - states[1:].to(DEV)) ** 2).backward()
        runs.append({"mean0": mean0.grad.clone(), **{k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}})
    assert set(runs[0]) == set(runs[1])
    differing = [k for k in runs[0] if not torch.equal(runs[0][k], runs[1][k])]
    assert not differing, f"gradients differ between two identical runs: {differing[:5]}"


@pytest.mark.gpu
def test_trainable_dynamics_keep_the_generic_path():
    from multimodalfilter_b200 import ops

    T, N, sd = 4, 8, 3
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=71)
    m = fill_parameters(M.DoorCrossmodalKalmanFilter(), seed=72).to(DEV).train()
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(DEV).contiguous()
    m.initialize_beliefs(mean=states[0].to(DEV), covariance=cov)
    ops.PROFILE.reset(enabled=True)
    est = m.forward_loop(observations={k: v[1:].to(DEV) for k, v in obs.items()}, controls=controls[1:].to(DEV))
    torch.mean((est - states[1:].to(DEV)) ** 2).backward()
    kernels = ops.PROFILE.collect()["kernels"]
    ops.PROFILE.reset()
    assert "ekf_loop_train" not in kernels and "ekf_loop_bwd" not in kernels, kernels
    assert any(p.grad is not None for p in m.filter_models[0].dynamics_model.parameters())


@pytest.mark.gpu
def test_train_e2e_runs_the_fused_ekf_step():
    """train_e2e (ref: crossmodal/train_helpers.py:124-162) restated call for call on a Kalman model with the curriculum's
    frozen dynamics: the loss goes down, the fused EKF kernels ran, the dynamics got no gradient and the virtual
    sensor's image encoder did."""
    import multimodalfilter_b200.fannypack as fannypack
    import multimodalfilter_b200.torchfilter as torchfilter_mmf
    from multimodalfilter_b200 import ops
    from multimodalfilter_b200.torchfilter.types import TrajectoryNumpy

    torch.manual_seed(0)
    model = fill_parameters(M.DoorCrossmodalKalmanFilter(), seed=3)
    buddy = fannypack.utils.Buddy("glue_e2e_kf", model, device="cuda:0")
    for f in model.filter_models:
        fannypack.utils.freeze_module(f.dynamics_model)
    s, o, c = synthetic_trajectories(17, 32, 3, seed=5)
    trajectories = [TrajectoryNumpy(s[:, n].numpy(), {k: v[:, n].numpy() for k, v in o.items()}, c[:, n].numpy())
                    for n in range(32)]

    def train_e2e(*, subsequence_length, epochs, batch_size=32, initial_cov_scale=0.1, measurement_initialize=False,
                  optimizer_name="train_filter_recurrent"):
        model.train()
        dataloader = torch.utils.data.DataLoader(
            torchfilter_mmf.data.SubsequenceDataset(trajectories=trajectories, subsequence_length=subsequence_length),
            batch_size=batch_size, shuffle=True, num_workers=0, drop_last=True)
        initial_covariance = torch.eye(model.state_dim, device=buddy.device) * initial_cov_scale
        return [torchfilter_mmf.train.train_filter(buddy, model, dataloader, initial_covariance=initial_covariance,
                                                   measurement_initialize=measurement_initialize,
                                                   optimizer_name=optimizer_name) for _ in range(epochs)]

    ops.PROFILE.reset(enabled=True)
    losses = train_e2e(subsequence_length=16, epochs=6, batch_size=16)
    kernels = ops.PROFILE.collect()["kernels"]
    ops.PROFILE.reset()
    steps = buddy.optimizer_steps
    assert steps == 6 * 4
    assert kernels["ekf_loop_train"]["count"] == steps and kernels["ekf_loop_bwd"]["count"] == steps, kernels
    assert np.isfinite(losses).all() and losses[-1] < losses[0], losses
    assert all(p.grad is None for f in model.filter_models for p in f.dynamics_model.parameters())
    assert any(p.grad is not None and p.grad.abs().sum() > 0 for n, p in model.named_parameters()
               if "virtual_sensor_model" in n and "image" in n), "the virtual sensor's image encoder received no gradient"
