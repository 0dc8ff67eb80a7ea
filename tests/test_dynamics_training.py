"""Training the dynamics models through the rollout kernels: ``training.FusedDynamicsRollout`` (mmf_dyn_rollout_fwd records
the tape, mmf_dyn_rollout_bwd walks the reverse recurrence from t = T-1 to 0), the eval rollout, and the dispatch of
``DynamicsModel.forward_loop`` / ``train_dynamics_single_step``.

CPU: the reverse recurrence, restated in float64 torch the way the kernel computes it, against torch.autograd through the
oracle's dynamics; the dispatch checks that need no device.
GPU: the eval rollout and the whole training path against the generic fp32 loop and the float64 oracle; the backward
kernel against a float64 backprop fed the kernel's own tape; freezing, chaining, determinism, NaN-prefilled raw entry
points and the two dynamics pre-training curricula."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import crossmodal_port as port  # installs the oracle shims on sys.path

from multimodalfilter_b200 import fused, training  # noqa: E402
from multimodalfilter_b200.crossmodal import models as M  # noqa: E402
from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories  # noqa: E402

DEV = "cuda:0"
f64 = torch.float64
U = 64
CLASSES = [("PushDynamicsModel", 2), ("DoorDynamicsModel", 3), ("DoorDynamicsModelBrent", 3)]
# mmf_pf_heads_weight_grads reduces with split-bf16 (hi + lo) operands: about 2^-16 relative per product, so the
# fused parameter gradients may exceed twice the generic fp32 error by this much (relative L2 against float64).
# Measured on a B200: the largest fused error over all parameters of the three models is 3.8e-7.
GRAD_FLOOR = 3e-5


# ---- the reverse recurrence, restated ---------------------------------------------------------------------------
def _layers(spec):
    """The 64x64 layers of the state chain in evaluation order: (Linear, 'first' | 'second' | 'mid')."""
    (_, pre), (mid, post, _) = spec.state, spec.shared
    layers = []
    for r in pre:
        layers += [(r.block1, "first"), (r.block2, "second")]
    layers.append((mid, "mid"))
    for r in post:
        layers += [(r.block1, "first"), (r.block2, "second")]
    return layers


def restated_forward(spec, x0, rows):
    """The rollout with its tape: x0 (N,sd), rows (T,N,64) -> states (T,N,sd), tape (T, L+1, N, 64), plane l = the input
    of 64x64 layer l, plane L = the input of the output layer."""
    in_lin, out = spec.state[0], spec.shared[2]
    sd = x0.shape[1]
    x, states, tape = x0, [], []
    for t in range(rows.shape[0]):
        h = torch.relu(x @ in_lin.weight.T + in_lin.bias)
        planes = []
        for lin, kind in _layers(spec):
            planes.append(h)
            if kind == "mid":
                h = h @ lin.weight[:, U:].T + rows[t]
            elif kind == "first":
                block_in, h = h, torch.relu(h @ lin.weight.T + lin.bias)
            else:
                h = torch.relu(h @ lin.weight.T + lin.bias + block_in)
        planes.append(h)
        y = h @ out.weight.T + out.bias
        x = x + y[:, :sd] * torch.sigmoid(y[:, sd:])
        states.append(x)
        tape.append(torch.stack(planes))
    return torch.stack(states), torch.stack(tape)


def restated_reverse(spec, tape, d_states):
    """k_dyn_rollout_bwd's recurrence: every ReLU mask from the tape (layer s's output is plane s+1, the input layer's is
    plane 0), y recomputed from plane L.  -> d_x0 (N,sd), delta (T, L+1, N, 64) (plane L = the input layer), d_y (T,N,sd+1)."""
    in_lin, out = spec.state[0], spec.shared[2]
    layers = _layers(spec)
    L = len(layers)
    T, _, N, _ = tape.shape
    sd = d_states.shape[-1]
    xb = d_states.new_zeros(N, sd)
    deltas, d_ys = [None] * T, [None] * T
    for t in reversed(range(T)):
        a = tape[t]
        y = a[L] @ out.weight.T + out.bias
        xb = xb + d_states[t]
        g = torch.sigmoid(y[:, sd:])
        yb = torch.cat([xb * g, g * (1 - g) * (xb * y[:, :sd]).sum(1, keepdim=True)], dim=1)
        grad = yb @ out.weight
        delta, resid = [None] * (L + 1), None
        for s in reversed(range(L)):
            lin, kind = layers[s]
            d = grad if kind == "mid" else grad * (a[s + 1] > 0)
            delta[s] = d
            grad = d @ (lin.weight[:, U:] if kind == "mid" else lin.weight)
            if kind == "second":
                resid = d
            elif kind == "first":
                grad = grad + resid
        delta[L] = grad * (a[0] > 0)
        xb = xb + delta[L] @ in_lin.weight
        deltas[t], d_ys[t] = torch.stack(delta), yb
    return xb, torch.stack(deltas), torch.stack(d_ys)


def restated_chain_grads(spec, x_in, tape, deltas, d_y):
    """Parameter gradients of the state chain in ``training.head_parameters`` order (mid Linear: state half only)."""
    L = tape.shape[1] - 1
    a = tape.transpose(0, 1).reshape(L + 1, -1, U)
    d = deltas.transpose(0, 1).reshape(L + 1, -1, U)
    grads = [d[L].T @ x_in, d[L].sum(0)]
    for s, (lin, kind) in enumerate(_layers(spec)):
        if kind == "mid":
            w = torch.zeros_like(lin.weight)
            w[:, U:] = d[s].T @ a[s]
            grads.append(w)
        else:
            grads += [d[s].T @ a[s], d[s].sum(0)]
    dy = d_y.reshape(-1, d_y.shape[-1])
    return grads + [dy.T @ a[L], dy.sum(0)]


def _mid_index(spec):
    return training.mid_layer_index(spec)


@pytest.mark.parametrize("cls,sd", CLASSES[:2])
@pytest.mark.parametrize("T", [1, 17])
@pytest.mark.parametrize("intermediate", [True, False])
def test_reverse_recurrence_restatement_equals_autograd_through_the_oracle(cls, sd, T, intermediate):
    g = torch.Generator().manual_seed(10 * sd + T)
    dyn = fill_parameters(getattr(port, cls)(), seed=3 + T).double()
    spec = fused._DynamicsSpec(dyn)
    assert spec.ok
    N, cd = 5, 7
    x0 = torch.randn(N, sd, generator=g, dtype=f64).requires_grad_(True)
    u = torch.randn(T, N, cd, generator=g, dtype=f64).requires_grad_(True)
    d_states = torch.randn(T, N, sd, generator=g, dtype=f64)
    if not intermediate:
        d_states[:-1] = 0.0  # a loss on the last state only
    states, _ = dyn.forward_loop(initial_states=x0, controls=u)
    params = [p for p in dyn.parameters() if p.requires_grad]
    want = torch.autograd.grad((states * d_states).sum(), [x0, u] + params)

    mid = spec.shared[0]
    rows = F.linear(dyn.control_layers(u.reshape(T * N, cd)), mid.weight[:, :U], mid.bias).reshape(T, N, U)
    st, tape = restated_forward(spec, x0.detach(), rows.detach())
    assert float((st - states).detach().abs().max()) <= 1e-12
    d_x0, deltas, d_y = restated_reverse(spec, tape, d_states)
    x_in = torch.cat([x0.detach()[None], st[:-1]]).reshape(T * N, sd)
    got = {id(p): gr for p, gr in zip(training.head_parameters(spec), restated_chain_grads(spec, x_in, tape, deltas, d_y))}
    row_inputs = [u] + list(dyn.control_layers.parameters()) + [mid.weight, mid.bias]
    for p, gr in zip(row_inputs, torch.autograd.grad(rows, row_inputs, deltas[:, _mid_index(spec)])):
        got[id(p)] = got[id(p)] + gr if id(p) in got else gr
    names = ["x0", "controls"] + [n for n, p in dyn.named_parameters() if p.requires_grad]
    for name, tensor, b in zip(names, [x0, u] + params, want):
        a = d_x0 if tensor is x0 else got[id(tensor)]
        rel = float(((a - b).norm() / b.norm().clamp_min(1e-300)).detach())
        assert rel <= 1e-10, f"{name}: relative error {rel:.3e}"


# ---- dispatch (no device needed) ----------------------------------------------------------------------------------
def test_dispatch_structure():
    dyn = M.DoorDynamicsModel()
    ctrl = torch.zeros(4, 8, 7)
    assert training.dynamics_structure_ok(dyn, ctrl)
    assert not training.dynamics_structure_ok(dyn, {"u": ctrl}), "dict controls keep the generic path"
    assert not training.dynamics_structure_ok(dyn, ctrl[:0]), "T = 0 keeps the generic path"
    dyn.fused_train = False
    assert not training.dynamics_structure_ok(dyn, ctrl)
    dyn.fused_train = True
    for module, kind in ((dyn.state_layers[0], "register_forward_hook"), (dyn, "register_forward_pre_hook"),
                         (dyn.shared_layers[2].block1, "register_forward_hook")):
        handle = getattr(module, kind)(lambda *a: None)
        assert not training.dynamics_structure_ok(dyn, ctrl), f"a hook ({kind}) keeps the generic path"
        handle.remove()
    assert training.dynamics_structure_ok(dyn, ctrl)

    class Odd(M.tf_base.DynamicsModel):
        def forward(self, *, initial_states, controls):
            return initial_states + controls[:, :1], None

    assert not training.dynamics_structure_ok(Odd(state_dim=1), ctrl), "unrecognised dynamics keep the generic path"


def test_cpu_tensors_keep_the_generic_loop():
    T, N, sd = 5, 6, 3
    dyn = fill_parameters(M.DoorDynamicsModelBrent(), seed=4)
    x0, u = torch.randn(N, sd), torch.randn(T, N, 7)
    assert training.dynamics_rollout(dyn, x0, u) is None
    states, trils = dyn.forward_loop(initial_states=x0, controls=u)
    x, want = x0, []
    for t in range(T):
        x, tril = dyn(initial_states=x, controls=u[t])
        want.append(x)
    assert torch.equal(states, torch.stack(want)) and torch.equal(trils, torch.stack([tril] * T))


# ---- GPU ----------------------------------------------------------------------------------------------------------
def _models(cls, seed):
    """(fused product model, generic product model, float64 oracle), identical parameters, all on the GPU."""
    fused_m = fill_parameters(getattr(M, cls)(), seed=seed).to(DEV)
    generic = fill_parameters(getattr(M, cls)(), seed=seed).to(DEV)
    generic.fused_train = False
    oracle = fill_parameters(getattr(port, cls)(), seed=seed).to(DEV, f64)
    return fused_m, generic, oracle


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300))


@pytest.mark.gpu
@pytest.mark.parametrize("cls,sd", CLASSES)
def test_eval_rollout_matches_generic_and_float64(cls, sd):
    from multimodalfilter_b200 import ops

    fused_m, generic, oracle = _models(cls, seed=11)
    for N in (1, 33, 4096):
        for T in (1, 15, 100):
            g = torch.Generator().manual_seed(N + T)
            x0 = torch.randn(N, sd, generator=g).to(DEV)
            u = torch.randn(T, N, 7, generator=g).to(DEV)
            with torch.no_grad():
                ops.PROFILE.reset(enabled=True)
                s_f, q_f = fused_m.forward_loop(initial_states=x0, controls=u)
                prof = ops.PROFILE.collect()
                ops.PROFILE.reset()
                s_g, q_g = generic.forward_loop(initial_states=x0, controls=u)
                s_r, _ = oracle.forward_loop(initial_states=x0.double(), controls=u.double())
            assert prof["launches"] == 1 and prof["kernels"]["dyn_rollout"]["count"] == 1, prof
            assert torch.equal(q_f, q_g)
            e_f, e_g = _rel(s_f, s_r), _rel(s_g, s_r)
            assert e_f <= 2 * e_g + 1e-6, f"N={N} T={T}: fused {e_f:.2e} vs generic {e_g:.2e}"


def _plan_of(dyn):
    plan = training._dynamics_plan(dyn)
    assert plan
    return plan


def _rows(dyn, u):
    spec = _plan_of(dyn).dyns[0]
    T, N, cd = u.shape
    mid = spec.shared[0]
    return F.linear(dyn.control_layers(u.reshape(T * N, cd)), mid.weight[:, :U], mid.bias).reshape(T, N, U)


@pytest.mark.gpu
@pytest.mark.parametrize("cls,sd", CLASSES[:2])
def test_tape_forward_is_bit_identical_to_the_eval_rollout(cls, sd):
    dyn = fill_parameters(getattr(M, cls)(), seed=12).to(DEV)
    plan = _plan_of(dyn)
    for N, T in ((1, 1), (33, 17), (4133, 15)):
        g = torch.Generator().manual_seed(N)
        x0 = torch.randn(N, sd, generator=g).to(DEV)
        u = torch.randn(T, N, 7, generator=g).to(DEV)
        with torch.no_grad():
            rows = _rows(dyn, u)
            states = plan.rollout(x0, rowbias=rows)
            s_t, act = plan.rollout_train(x0, rows)
        assert torch.equal(states, s_t), (N, T)
        assert torch.isfinite(act).all()


@pytest.mark.gpu
@pytest.mark.parametrize("cls,sd", CLASSES[:2])
@pytest.mark.parametrize("N", [37, 5003])
@pytest.mark.parametrize("T", [1, 17])
def test_backward_kernel_matches_float64_given_the_tape(cls, sd, N, T):
    """N = 5003 over 148 SMs: 32 warps per CTA, not a divisor of N, and a second trajectory for some warps."""
    from multimodalfilter_b200 import ops

    dyn = fill_parameters(getattr(M, cls)(), seed=13).to(DEV)
    plan = _plan_of(dyn)
    g = torch.Generator().manual_seed(N * T)
    x0 = torch.randn(N, sd, generator=g).to(DEV)
    u = torch.randn(T, N, 7, generator=g).to(DEV)
    d_states = torch.randn(T, N, sd, generator=g).to(DEV)
    with torch.no_grad():
        _, act = plan.rollout_train(x0, _rows(dyn, u))
        delta, d_y, d_x0 = ops.dyn_rollout_bwd(plan.structs[0].dynamics, T, N, act, d_states)
        spec64 = fused._DynamicsSpec(fill_parameters(getattr(M, cls)(), seed=13).to(DEV, f64))
        tape = ops.rows_view(act).double().view(-1, T, N, U).transpose(0, 1)  # (T, L+1, N, 64)
        want_x0, want_delta, want_dy = restated_reverse(spec64, tape, d_states.double())
    got_delta = ops.rows_view(delta).view(-1, T, N, U).transpose(0, 1)
    assert _rel(d_x0, want_x0) <= 1e-6, f"d_x0 {_rel(d_x0, want_x0):.2e}"
    assert _rel(d_y.view(T, N, sd + 1), want_dy) <= 1e-6, f"d_y {_rel(d_y.view(T, N, sd + 1), want_dy):.2e}"
    for l in range(delta.shape[0]):
        rel = _rel(got_delta[:, l], want_delta[:, l])
        assert rel <= 1e-6, f"delta plane {l}: relative L2 {rel:.2e}"


def _train_run(dyn, x0, u, target, *, x0_grad=False, u_grad=False):
    x0 = x0.clone().requires_grad_(x0_grad)
    u = u.clone().requires_grad_(u_grad)
    states, _ = dyn.forward_loop(initial_states=x0, controls=u)
    loss = torch.mean((states - target) ** 2)
    loss.backward()
    grads = {k: p.grad.detach().double().cpu() for k, p in dyn.named_parameters() if p.grad is not None}
    if x0_grad:
        grads["x0"] = x0.grad.double().cpu()
    if u_grad:
        grads["controls"] = u.grad.double().cpu()
    return float(loss), grads


def _data(T, N, sd, seed):
    states, _, controls = synthetic_trajectories(T + 1, N, sd, seed=seed)
    return states[0].to(DEV), controls[1:].to(DEV), states[1:].to(DEV)


@pytest.mark.gpu
@pytest.mark.parametrize("cls,sd", CLASSES)
def test_training_gradients_fused_vs_generic_vs_float64(cls, sd):
    from multimodalfilter_b200 import ops

    T, N = 15, 32
    x0, u, target = _data(T, N, sd, seed=21)
    fused_m, generic, oracle = _models(cls, seed=22)
    ops.PROFILE.reset(enabled=True)
    l_f, g_f = _train_run(fused_m, x0, u, target, x0_grad=True, u_grad=True)
    kernels = ops.PROFILE.collect()["kernels"]
    ops.PROFILE.reset()
    assert kernels["dyn_rollout_train"]["count"] == 1 and kernels["dyn_rollout_bwd"]["count"] == 1, kernels
    l_g, g_g = _train_run(generic, x0, u, target, x0_grad=True, u_grad=True)
    l_r, g_r = _train_run(oracle, x0.double(), u.double(), target.double(), x0_grad=True, u_grad=True)
    assert set(g_f) == set(g_g) == set(g_r) and {"x0", "controls", "shared_layers.0.weight"} <= set(g_r)
    assert abs(l_f - l_r) <= 2 * abs(l_g - l_r) + 1e-6 * abs(l_r), (l_f, l_g, l_r)
    worst = 0.0
    for k in g_r:
        e_f, e_g = _rel(g_f[k], g_r[k]), _rel(g_g[k], g_r[k])
        worst = max(worst, e_f)
        assert e_f <= 2 * e_g + GRAD_FLOOR, f"{k}: fused {e_f:.2e} vs generic {e_g:.2e} (relative to float64)"
    print(f"{cls}: largest fused relative L2 error {worst:.2e}")


def _compare(g_a, g_b, bar=GRAD_FLOOR):
    assert set(g_a) == set(g_b), (sorted(g_a), sorted(g_b))
    for k in g_b:
        assert _rel(g_a[k], g_b[k]) <= bar, f"{k}: relative L2 {_rel(g_a[k], g_b[k]):.2e}"


@pytest.mark.gpu
def test_partial_freezing():
    T, N, sd = 15, 32, 3
    x0, u, target = _data(T, N, sd, seed=31)
    fused_m, generic, _ = _models("DoorDynamicsModel", seed=32)
    for m in (fused_m, generic):
        for p in m.state_layers.parameters():
            p.requires_grad_(False)
    _, g_f = _train_run(fused_m, x0, u, target)
    _, g_g = _train_run(generic, x0, u, target)
    assert all(p.grad is None for p in fused_m.state_layers.parameters())
    assert not any(k.startswith("state_layers") for k in g_f)
    _compare(g_f, g_g, bar=1e-4)

    fused_m, generic, _ = _models("DoorDynamicsModel", seed=33)
    for m in (fused_m, generic):
        for p in m.parameters():
            p.requires_grad_(False)
    _, g_f = _train_run(fused_m, x0, u, target, x0_grad=True)
    _, g_g = _train_run(generic, x0, u, target, x0_grad=True)
    assert set(g_f) == {"x0"}
    _compare(g_f, g_g, bar=1e-5)


@pytest.mark.gpu
def test_second_rollout_chains_the_gradient_into_the_first():
    from multimodalfilter_b200 import ops

    T, N, sd = 8, 16, 2
    x0, u, target = _data(2 * T, N, sd, seed=41)
    results = []
    for split in (False, True):
        dyn = fill_parameters(M.PushDynamicsModel(), seed=42).to(DEV)
        x = x0.clone().requires_grad_(True)
        ops.PROFILE.reset(enabled=True)
        if split:
            a, _ = dyn.forward_loop(initial_states=x, controls=u[:T])
            b, _ = dyn.forward_loop(initial_states=a[-1], controls=u[T:])
            states = torch.cat([a, b])
        else:
            states, _ = dyn.forward_loop(initial_states=x, controls=u)
        torch.mean((states - target) ** 2).backward()
        kernels = ops.PROFILE.collect()["kernels"]
        ops.PROFILE.reset()
        assert kernels["dyn_rollout_bwd"]["count"] == (2 if split else 1), kernels
        results.append({"x0": x.grad.double().cpu(), **{k: p.grad.double().cpu() for k, p in dyn.named_parameters()
                                                          if p.grad is not None}})
    _compare(results[1], results[0], bar=1e-4)


@pytest.mark.gpu
def test_backward_is_bit_reproducible():
    T, N, sd = 15, 4096, 3
    x0, u, target = _data(T, N, sd, seed=51)
    runs = []
    for _ in range(2):
        dyn = fill_parameters(M.DoorDynamicsModelBrent(), seed=52).to(DEV)
        runs.append(_train_run(dyn, x0, u, target, x0_grad=True, u_grad=True)[1])
    differing = [k for k in runs[0] if not torch.equal(runs[0][k], runs[1][k])]
    assert set(runs[0]) == set(runs[1]) and not differing, differing


@pytest.mark.gpu
def test_raw_entry_points_write_every_element():
    from multimodalfilter_b200 import _lib

    lib = _lib.load()
    dyn = fill_parameters(M.DoorDynamicsModel(), seed=61).to(DEV)
    plan = _plan_of(dyn)
    plan.refresh(torch.device(DEV))
    chain, rows_struct = plan.structs[0].dynamics, plan.structs[0].dynamics_rows
    T, N, sd, L = 17, 301, 3, 9
    g = torch.Generator().manual_seed(62)
    x0 = torch.randn(N, sd, generator=g).to(DEV)
    u = torch.randn(T, N, 7, generator=g).to(DEV)
    nan = lambda *shape: torch.full(shape, float("nan"), device=DEV)  # noqa: E731
    with torch.no_grad():
        rows = _rows(dyn, u).contiguous()
    stream = _lib.stream_of(x0)
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    for via_rows in (True, False):
        states, act = nan(T, N, sd), nan(L + 1, 16, T * N, 4)
        _lib.check(lib.mmf_dyn_rollout_fwd(C.byref(chain), C.byref(rows_struct), T, N, ptr(x0), ptr(u),
                                           ptr(rows) if via_rows else None, ptr(states), ptr(act), stream))
        torch.cuda.synchronize()
        assert torch.isfinite(states).all() and torch.isfinite(act).all(), via_rows
    for d_states in (torch.randn(T, N, sd, generator=g).to(DEV), None):
        delta, d_y, d_x0 = nan(L + 1, 16, T * N, 4), nan(T * N, sd + 1), nan(N, sd)
        _lib.check(lib.mmf_dyn_rollout_bwd(C.byref(chain), T, N, ptr(act), ptr(d_states), ptr(delta), ptr(d_y),
                                           ptr(d_x0), stream))
        torch.cuda.synchronize()
        assert torch.isfinite(delta).all() and torch.isfinite(d_y).all() and torch.isfinite(d_x0).all()
        if d_states is None:
            assert not delta.any() and not d_y.any() and not d_x0.any()
    assert lib.mmf_dyn_rollout_fwd(C.byref(chain), None, T, N, ptr(x0), ptr(u), None, ptr(states), None, stream) != 0, \
        "without rowbias the control rows are required"


@pytest.mark.gpu
@pytest.mark.parametrize("phase", ["single_step", "recurrent"])
def test_dynamics_curricula_run_the_fused_kernels(phase):
    """train_pf_dynamics_single_step / train_pf_dynamics_recurrent (ref: crossmodal/train_helpers.py:30-73) restated call
    for call: SingleStepDataset / SubsequenceDataset(subsequence_length=16) -> DataLoader(batch_size=32, shuffle=True) ->
    torchfilter.train.train_dynamics_single_step / train_dynamics_recurrent.  The loss is recorded per step, so the first
    step can be compared with the generic path's."""
    import multimodalfilter_b200.fannypack as fannypack
    import multimodalfilter_b200.torchfilter as torchfilter_mmf
    from multimodalfilter_b200 import ops
    from multimodalfilter_b200.torchfilter.types import TrajectoryNumpy

    s, o, c = synthetic_trajectories(33, 64, 2, seed=71)
    trajectories = [TrajectoryNumpy(s[:, n].numpy(), {k: v[:, n].numpy() for k, v in o.items()}, c[:, n].numpy())
                    for n in range(64)]

    def run(fused_train):
        torch.manual_seed(0)
        model = fill_parameters(M.PushCrossmodalParticleFilter(), seed=72)
        dynamics_model = model.dynamics_model
        dynamics_model.fused_train = fused_train
        buddy = fannypack.utils.Buddy(f"dyn_{phase}_{fused_train}", model, device=DEV)
        losses = []

        def mse(pred, target):
            loss = F.mse_loss(pred, target)
            losses.append(float(loss.detach()))
            return loss

        for _ in range(3):
            if phase == "single_step":
                dataloader = torch.utils.data.DataLoader(torchfilter_mmf.data.SingleStepDataset(trajectories=trajectories),
                                                         batch_size=32, shuffle=True, num_workers=0)
                torchfilter_mmf.train.train_dynamics_single_step(buddy, dynamics_model, dataloader, loss_function=mse)
            else:
                dataloader = torch.utils.data.DataLoader(
                    torchfilter_mmf.data.SubsequenceDataset(trajectories=trajectories, subsequence_length=16),
                    batch_size=32, shuffle=True, num_workers=0)
                torchfilter_mmf.train.train_dynamics_recurrent(buddy, dynamics_model, dataloader, loss_function=mse)
        return losses, buddy.optimizer_steps

    ops.PROFILE.reset(enabled=True)
    losses, steps = run(True)
    kernels = ops.PROFILE.collect()["kernels"]
    ops.PROFILE.reset()
    assert kernels["dyn_rollout_train"]["count"] == steps and kernels["dyn_rollout_bwd"]["count"] == steps, kernels
    assert np.isfinite(losses).all() and np.mean(losses[-5:]) < np.mean(losses[:5]), losses
    generic, _ = run(False)
    assert abs(losses[0] - generic[0]) <= 1e-5 * abs(generic[0]), (losses[0], generic[0])
