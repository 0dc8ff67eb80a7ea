"""Training the per-trajectory MLP stacks through the row-program kernels: ``training.FusedRowProgram``
(mmf_row_mlp_train_fwd records the tape, mmf_row_mlp_bwd walks the host-compiled reverse program,
mmf_row_mlp_weight_grads reduces dW / db), the reverse compiler of ``fused.RowProgram`` and the dispatch of the four
callers (weight models, virtual sensors, PF head features, the M = 1 head).

CPU: a float64 interpreter of the compiled forward and reverse op lists against torch autograd through the same modules,
with every delta-slot read checked against the value that must be there; the dispatch decisions that need no device.
GPU: the kernels against the eval launch (bit-identical), against a float64 backprop fed the kernel's own tape, run to
run, with NaN-prefilled outputs; one step of each training phase against the torch path and float64."""
import copy

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import crossmodal_port as port  # noqa: F401  (installs the oracle shims on sys.path)

from multimodalfilter_b200 import _lib, fused, ops  # noqa: E402
from multimodalfilter_b200.crossmodal import models as M  # noqa: E402
from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories  # noqa: E402

DEV = "cuda:0"
f64 = torch.float64
U = 64
SUBSETS = [{"image"}, {"pos"}, {"sensors"}, {"pos", "sensors"}, {"image", "pos"}, {"image", "sensors"},
           {"image", "pos", "sensors"}]


# ---- the model zoo's programs, and torch restatements of what each computes ----------------------------------------
def _feats(m, ins):
    return [x if mod == "image" else enc(x) for (mod, enc), x in zip(m._encoder_list(), ins)]


def zoo():
    """(name, owner module, program, torch function of the program's inputs -> list of outputs)."""
    cases = []
    for cls in (M.PushCrossmodalWeightModel, M.DoorCrossmodalWeightModel):
        m = fill_parameters(cls(know_image_blackout=False), seed=3)
        cases.append((cls.__name__, m, m.program(), lambda m, ins: [m.fusion_layers(torch.cat(_feats(m, ins), 1))]))
    for cls, sd in ((M.PushCrossmodalKalmanFilterWeightModel, 2), (M.DoorCrossmodalKalmanFilterWeightModel, 3)):
        m = fill_parameters(cls(state_dim=sd), seed=4)
        cases.append((cls.__name__, m, m.program(), lambda m, ins: [m.fusion_layers(torch.cat(_feats(m, ins), 1))]))

    def sensor(m, ins):
        h = m.shared_layers(torch.cat(_feats(m, ins), 1))
        return [m.z_layer(h[:, :U]), m.r_layer(h[:, U:])]

    for cls in (M.PushVirtualSensorModel, M.DoorVirtualSensorModel):
        for mods in SUBSETS:
            m = fill_parameters(cls(modalities=mods), seed=5)
            cases.append((f"{cls.__name__}{sorted(mods)}", m, m.program(), sensor))
    for cls, sd in ((M.PushMeasurementModel, 2), (M.DoorMeasurementModel, 3)):
        for mods in ({"pos", "sensors"}, {"image", "pos", "sensors"}):
            m = fill_parameters(cls(modalities=mods), seed=6)
            cases.append((f"{cls.__name__}{sorted(mods)}.features", m, fused._HeadSpec(m, sd)._feature_program(),
                          lambda m, ins: [torch.cat(_feats(m, ins), 1)]))
        for mods in ({"image"}, {"pos", "sensors"}):
            m = fill_parameters(cls(modalities=mods), seed=7)
            cases.append((f"{cls.__name__}{sorted(mods)}.single", m, m.single_program(),
                          lambda m, ins: [m.shared_layers(torch.cat(_feats(m, ins[:-1]) + [m.state_layers(ins[-1])], 1))]))
    return cases


ZOO = zoo()


def _inputs(prog, rows, seed, dtype=f64, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(rows, d, generator=g, dtype=f64).to(device, dtype) for d in prog.in_dims]


def _act(y, act):
    return torch.relu(y) if act == _lib.MLP_RELU else torch.sigmoid(y) if act == _lib.MLP_SIGMOID else y


# ---- float64 interpreter of the compiled op lists ------------------------------------------------------------------
def interpret(prog, rev, inputs, d_outs, tape=None):
    """Forward and reverse program in float64 over (rows, slots) matrices.  ``tape``: per op (x, y) to use instead of
    the interpreter's own forward (a backprop fed the kernel's tape).  Every read of a delta slot asserts that the slot
    holds the delta of the value the reverse program means to read (no slot is read after another value overwrote it).
    -> outputs, d_inputs (by rev.inputs), per op (g, dW, db)."""
    values, reads, out_spans = prog.trace()
    n_in = len(prog.in_slots)
    rows = inputs[0].shape[0]
    W = [(lin.weight.detach().double().cpu(), lin.bias.detach().double().cpu()) for lin in prog.params]
    S = torch.zeros(rows, prog.scratch, dtype=f64)
    for x, s, d in zip(inputs, prog.in_slots, prog.in_dims):
        S[:, s:s + d] = x
    own = []
    for o, op in enumerate(prog.ops):
        x = S[:, op.src:op.src + op.in_dim].clone()
        y = x @ W[o][0].t() + W[o][1]
        if op.res >= 0:
            y = y + S[:, op.res:op.res + op.out_dim]
        y = _act(y, op.act)
        own.append((x, y))
        S[:, op.dst:op.dst + op.out_dim] = y
    outs = [S[:, s:s + d].clone() for s, d in zip(prog.out_slots, prog.out_dims)]
    tape = tape or own

    D = torch.full((rows, rev.scratch), float("nan"), dtype=f64)
    tag = [None] * rev.scratch

    def write(slot, span, val, acc):
        if acc:
            assert tag[slot:slot + len(span)] == list(span), "accumulating into a slot that holds another value"
            val = D[:, slot:slot + len(span)] + val
        D[:, slot:slot + len(span)] = val
        tag[slot:slot + len(span)] = list(span)

    for sp, s, d in zip(out_spans, rev.dout_slots, d_outs):
        write(s, sp, d, False)
    per_op = {}
    for b in rev.ops:
        op = prog.ops[b.op]
        x, y = tape[b.op]
        assert tag[b.g:b.g + op.out_dim] == [(n_in + b.op, j) for j in range(op.out_dim)], f"op {b.op}: stale delta"
        g = D[:, b.g:b.g + op.out_dim]
        if op.act == _lib.MLP_RELU:
            g = g * (y > 0)
        elif op.act == _lib.MLP_SIGMOID:
            g = g * y * (1 - y)
        D[:, b.g:b.g + op.out_dim] = g
        src, res = reads[b.op]
        if b.dres >= 0:
            write(b.dres, res, g, bool(b.flags & _lib.MLP_DRES_ACC))
        if b.dsrc >= 0:
            write(b.dsrc, src, g @ W[b.op][0], bool(b.flags & _lib.MLP_DSRC_ACC))
        per_op[b.op] = (g.clone(), g.t() @ x, g.sum(0))
    d_in = []
    for i, s in zip(rev.inputs, rev.din_slots):
        assert tag[s:s + prog.in_dims[i]] == [(i, k) for k in range(prog.in_dims[i])], f"input {i}: stale delta"
        d_in.append(D[:, s:s + prog.in_dims[i]].clone())
    return outs, d_in, per_op


@pytest.mark.parametrize("case", range(len(ZOO)), ids=[c[0] for c in ZOO])
@pytest.mark.parametrize("need", ["all", "first"])
def test_reverse_program_matches_autograd_float64(case, need):
    name, m, prog, fn = ZOO[case]
    assert prog is not None, f"{name}: not fusable"
    m = copy.deepcopy(m).double()
    prog = copy.deepcopy(prog)
    prog.params = [dict(m.named_modules())[n] for n in _param_names(ZOO[case][1], ZOO[case][2])]
    rows = 5
    ins = _inputs(prog, rows, seed=case)
    g = torch.Generator().manual_seed(100 + case)
    d_outs = [torch.randn(rows, d, generator=g, dtype=f64) for d in prog.out_dims]
    need_in = tuple(True for _ in ins) if need == "all" else tuple(i == 0 for i in range(len(ins)))
    rev = prog.reverse(need_in)
    outs, d_in, per_op = interpret(prog, rev, ins, d_outs)
    ins_t = [x.clone().requires_grad_(n) for x, n in zip(ins, need_in)]
    ref = fn(m, ins_t)
    for a, b in zip(outs, ref):
        torch.testing.assert_close(a, b.detach(), rtol=1e-10, atol=1e-10)
    params = prog.parameters()
    wrt = [x for x in ins_t if x.requires_grad] + params
    grads = torch.autograd.grad(ref, wrt, d_outs, allow_unused=True)
    g_in, g_par = grads[:len(wrt) - len(params)], grads[len(wrt) - len(params):]
    assert rev.inputs == [i for i, n in enumerate(need_in) if n]
    for a, b in zip(d_in, g_in):
        torch.testing.assert_close(a, b, rtol=1e-10, atol=1e-10)
    for o in range(len(prog.ops)):
        _, dW, db = per_op[o]
        torch.testing.assert_close(dW, g_par[2 * o], rtol=1e-10, atol=1e-10)
        torch.testing.assert_close(db, g_par[2 * o + 1], rtol=1e-10, atol=1e-10)


def _param_names(module, prog):
    names = {id(mod): n for n, mod in module.named_modules()}
    return [names[id(lin)] for lin in prog.params]


@pytest.mark.parametrize("case", range(len(ZOO)), ids=[c[0] for c in ZOO])
def test_reached_sets_follow_the_outputs(case):
    """Parameters reached from each output alone: the ops the output's value depends on (the z head alone leaves the r
    head's parameters without a gradient, as autograd through the modules does)."""
    name, m, prog, fn = ZOO[case]
    for k in range(len(prog.out_dims)):
        have = [i == k for i in range(len(prog.out_dims))]
        ops_reached, _ = prog.reached(have)
        ins = [x.requires_grad_(False) for x in _inputs(prog, 3, seed=1, dtype=torch.float32)]
        out = fn(m, ins)[k]
        used = torch.autograd.grad(out.sum(), prog.parameters(), allow_unused=True)
        want = {o for o in range(len(prog.ops)) if used[2 * o] is not None}
        assert ops_reached == want, name


# ---- dispatch (no device) ------------------------------------------------------------------------------------------
def test_training_dispatch_decisions():
    m = M.DoorVirtualSensorModel(modalities={"image"})
    assert fused.row_train_ok(m)  # grad mode on, flag on by default, no hooks, no per-row tensors to check
    with torch.no_grad():
        assert not fused.row_train_ok(m)
    m.fused_train = False
    assert not fused.row_train_ok(m)
    m.fused_train = True
    h = m.shared_layers[0].register_forward_hook(lambda *a: None)
    assert not fused.row_train_ok(m)
    h.remove()
    h = m.register_forward_pre_hook(lambda *a: None)
    assert not fused.row_train_ok(m)
    h.remove()
    assert fused.row_train_ok(m)
    assert not fused.row_train_ok(m, torch.zeros(4, 3))  # CPU rows
    assert not fused.row_train_ok(m, torch.zeros(4, 3, dtype=f64))
    assert not fused.row_train_ok(m, {"gripper_pos": torch.zeros(4, 3)})
    # the filters' switch governs their recursion only: it does not reach these modules
    kf = M.DoorCrossmodalKalmanFilter()
    kf.fused_train = False
    assert all(mod.fused_train for mod in kf.modules() if isinstance(mod, M._Encoders))


def test_reverse_feasibility_is_decided_when_the_path_is_chosen():
    """A stack whose reverse program does not compile keeps the torch modules under grad mode (the inference launch still
    takes it); a wide stack (units = 96: the shared Linear reads 384 inputs) is trainable."""
    lin = nn.Linear(3, 4)
    prog = fused.RowProgram()
    src = prog.input(3)
    out, dim = prog.sequential([lin], src, 3)
    prog.output(out, dim)
    prog.output(out, dim)  # two outputs of one value: no reverse program
    assert not prog.trainable()
    assert fused.usable(prog) is None
    with torch.no_grad():
        assert fused.usable(prog) is prog
    with pytest.raises(fused.NotFusable):
        prog.run_train([torch.zeros(2, 3)])
    for cls in (M.DoorMeasurementModel, M.PushMeasurementModel):
        wide = cls(units=96).single_program()
        assert max(op.in_dim for op in wide.ops) == 384 and wide.trainable() and fused.usable(wide) is wide


def test_not_fusable_stack_keeps_the_torch_modules():
    m = M.DoorCrossmodalWeightModel(know_image_blackout=False)
    m.fusion_layers = nn.Sequential(nn.Linear(3 * U, U), nn.Tanh(), nn.Linear(U, 2))
    assert m.program() is None
    obs = {"image": torch.randn(4, 32, 32), "gripper_pos": torch.randn(4, 3), "gripper_sensors": torch.randn(4, 7)}
    out = m(observations=obs)  # CPU tensors: the torch path, with autograd
    assert out.shape == (4, 2) and out.requires_grad


# ---- GPU: the kernels ----------------------------------------------------------------------------------------------
def _pass_rows(scratch):
    """Rows of one full pass of the row kernels' grid (warps per CTA from the shared-memory budget of the scratch: the
    forward scratch for k_row_mlp / k_row_mlp_train, the delta scratch for k_row_mlp_bwd)."""
    props = torch.cuda.get_device_properties(0)
    window = props.shared_memory_per_block_optin
    wtiles, per_warp = 2 * 64 * 64 * 4, 8 * scratch * 4
    fit = lambda b: min(16, max(0, (b - wtiles - 1024) // per_warp))  # noqa: E731
    w1, w2 = fit(window), fit(window // 2)
    per_sm, warps = (2, w2) if 2 * w2 >= w1 else (1, w1)
    return props.multi_processor_count * per_sm * warps * 8


KERNEL_CASES = [c for c in ZOO if c[0] in ("DoorVirtualSensorModel['image', 'pos', 'sensors']",
                                           "DoorCrossmodalKalmanFilterWeightModel", "PushCrossmodalWeightModel",
                                           "PushMeasurementModel['image', 'pos', 'sensors'].features",
                                           "DoorMeasurementModel['pos', 'sensors'].single")]


def _nan_empty(real):
    def empty(*size, **kw):
        t = real(*size, **kw)
        return t.fill_(float("nan")) if t.is_floating_point() else t.fill_(255)
    return empty


def _rel(a, b):
    return float((a.double() - b).abs().max() / max(float(b.abs().max()), 1e-30))


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["small", "pass", "large"])
def test_kernels_against_eval_launch_and_float64(which, monkeypatch):
    monkeypatch.setattr(torch, "empty", _nan_empty(torch.empty))  # every output of the raw entry points is NaN first
    assert len(KERNEL_CASES) == 5
    for name, m, prog, _ in KERNEL_CASES:
        m = m.to(DEV)
        w_fwd, w_t = prog.train_weights(torch.device(DEV))
        need = tuple(mod == "image" for mod, _ in m._encoder_list())[:len(prog.in_dims)]
        need = need + (False,) * (len(prog.in_dims) - len(need))
        need = need if any(need) else (True,) + need[1:]
        rev = prog.reverse(need)
        p, q = _pass_rows(prog.scratch), _pass_rows(rev.scratch)
        rows_list = {"small": [1, 7, 8, 9], "pass": sorted({p - 1, p, p + 1, q - 1, q, q + 1}),
                     "large": [61440, 122880]}[which]
        for rows in rows_list:
            ins = _inputs(prog, rows, seed=rows, dtype=torch.float32, device=DEV)
            ev = ops.row_mlp(prog.ops, w_fwd, ins, prog.in_slots, prog.out_dims, prog.out_slots, prog.scratch)
            tr, tape = ops.row_mlp_train_fwd(prog.ops, w_fwd, ins, prog.in_slots, prog.out_dims, prog.out_slots,
                                            prog.scratch)
            for a, b in zip(ev, tr):
                assert torch.equal(a, b), f"{name} rows={rows}: the tape launch changed the outputs"
            g = torch.Generator(device=DEV).manual_seed(rows)
            d_outs = [torch.randn(rows, d, generator=g, device=DEV) for d in prog.out_dims]
            runs = []
            for _ in range(2):
                d_in, delta = ops.row_mlp_bwd(prog.ops, w_t, tape, rev.ops, d_outs, rev.dout_slots,
                                              [prog.in_dims[i] for i in rev.inputs], rev.din_slots, rev.scratch)
                pack = ops.row_mlp_weight_grads(prog.ops, rows, tape, delta, prog._w_floats)
                runs.append((d_in, delta, pack))
            (d_in, delta, pack), (d_in2, delta2, pack2) = runs
            assert all(torch.equal(a, b) for a, b in zip(d_in + [delta, pack], d_in2 + [delta2, pack2])), \
                f"{name} rows={rows}: two runs differ"
            assert not torch.isnan(pack).any() and all(not torch.isnan(x).any() for x in d_in)
            # float64 backprop fed the kernel's own tape
            G = (rows + 7) // 8
            tf = sum(op.in_dim + op.out_dim for op in prog.ops)
            gf = sum(op.out_dim for op in prog.ops)
            tape_rows = tape.view(G, tf, 8).permute(0, 2, 1).reshape(G * 8, tf)[:rows].double().cpu()
            delta_rows = delta.view(G, gf, 8).permute(0, 2, 1).reshape(G * 8, gf)[:rows].double().cpu()
            kt, off = [], 0
            for op in prog.ops:
                kt.append((tape_rows[:, off:off + op.in_dim], tape_rows[:, off + op.in_dim:off + op.in_dim + op.out_dim]))
                off += op.in_dim + op.out_dim
            cpu_ins = [x.double().cpu() for x in ins]
            _, d_ref, per_op = interpret(prog, rev, cpu_ins, [d.double().cpu() for d in d_outs], tape=kt)
            for a, b in zip(d_in, d_ref):
                assert _rel(a.cpu(), b) <= 1e-6, f"{name} rows={rows}: d_input {_rel(a.cpu(), b):.2e}"
            goff = 0
            for o, op in enumerate(prog.ops):
                g_ref, dW_ref, db_ref = per_op[o]
                e = _rel(delta_rows[:, goff:goff + op.out_dim], g_ref)
                assert e <= 1e-6, f"{name} rows={rows} op {o}: delta plane {e:.2e}"
                goff += op.out_dim
                nw = op.out_dim * op.in_dim
                dW = pack[op.w_off:op.w_off + nw].view(op.out_dim, op.in_dim).cpu()
                db = pack[op.w_off + nw:op.w_off + nw + op.out_dim].cpu()
                assert _rel(dW, dW_ref) <= 1e-6 and _rel(db, db_ref) <= 1e-6, \
                    f"{name} rows={rows} op {o}: dW {_rel(dW, dW_ref):.2e} db {_rel(db, db_ref):.2e}"
        m.cpu()


# ---- GPU: one step of each training phase --------------------------------------------------------------------------
def set_row_flag(model, on):
    for mod in model.modules():
        if isinstance(mod, M._Encoders):
            mod.fused_train = on


def _grads(model):
    return {k: p.grad.detach().double().cpu() for k, p in model.named_parameters() if p.grad is not None}


def _step(make, run, on, device=DEV, dtype=torch.float32):
    model = make().to(device, dtype)
    set_row_flag(model, on)
    ops.PROFILE.reset(enabled=device == DEV)
    loss = run(model, device, dtype)
    loss.backward()
    kernels = ops.PROFILE.collect()["kernels"] if device == DEV else {}
    ops.PROFILE.reset()
    return float(loss), _grads(model), kernels


def compare(make, run, make_ref=None, floor=0.0):
    """One step with the row programs (flag on), with the torch modules (flag off) and in float64 on the CPU (``make_ref``:
    the oracle port's model with the same parameters, for filters whose recursion needs CUDA; default ``make``).  Loss
    and every parameter gradient of the fused step must be within twice the torch step's error against float64 (plus
    1e-5 relative, plus ``floor`` times the largest gradient for steps whose float64 reference differs in kind)."""
    l_on, g_on, k_on = _step(make, run, True)
    l_off, g_off, k_off = _step(make, run, False)
    for name in ("row_mlp_train", "row_mlp_bwd", "row_mlp_dw"):
        assert name in k_on, f"{name} did not run: {sorted(k_on)}"
        assert name not in k_off, f"{name} ran with the flag off"
    assert set(g_on) == set(g_off) and len(g_on) > 0
    l_ref, g_ref, _ = _step(make_ref or make, run, False, device="cpu", dtype=f64)
    assert set(g_ref) == set(g_on)
    assert abs(l_on - l_ref) <= 2 * abs(l_off - l_ref) + 1e-6 * abs(l_ref), (l_on, l_off, l_ref)
    big = max(float(g.norm()) for g in g_ref.values())
    for k in g_ref:
        scale = float(g_ref[k].norm()) or 1.0
        e_on, e_off = float((g_on[k] - g_ref[k]).norm()) / scale, float((g_off[k] - g_ref[k]).norm()) / scale
        assert e_on <= 2 * e_off + 1e-5 + floor * big / scale, \
            f"{k}: fused {e_on:.2e} vs torch {e_off:.2e} (relative to float64)"


def _obs(N, sd, seed, T=1):
    states, obs, controls = synthetic_trajectories(T, N, sd, seed=seed)
    return states, obs, controls


@pytest.mark.gpu
@pytest.mark.parametrize("cls,sd", [(M.DoorVirtualSensorModel, 3), (M.PushVirtualSensorModel, 2)])
@pytest.mark.parametrize("mods", [{"pos", "sensors"}, {"image"}])
def test_train_virtual_sensor_step(cls, sd, mods):
    states, obs, _ = _obs(64, sd, seed=11)

    def run(m, dev, dt):
        z, _ = m(observations={k: v[0].to(dev, dt) for k, v in obs.items()})
        return F.mse_loss(z, states[0].to(dev, dt))

    compare(lambda: fill_parameters(cls(modalities=mods), seed=12), run)


@pytest.mark.gpu
@pytest.mark.parametrize("cls,sd", [(M.PushMeasurementModel, 2), (M.DoorMeasurementModel, 3)])
@pytest.mark.parametrize("mods,units", [({"pos", "sensors"}, 64), ({"image"}, 64), ({"image", "pos", "sensors"}, 128)])
def test_train_particle_filter_measurement_step(cls, sd, mods, units):
    states, obs, _ = _obs(64, sd, seed=13)
    target = torch.randn(64, generator=torch.Generator().manual_seed(14))

    def run(m, dev, dt):
        pred = m(states=states[0].to(dev, dt)[:, None, :], observations={k: v[0].to(dev, dt) for k, v in obs.items()})
        assert pred.shape == (64, 1)
        return F.mse_loss(pred[:, 0], target.to(dev, dt))

    compare(lambda: fill_parameters(cls(units=units, modalities=mods), seed=15), run)


@pytest.mark.gpu
@pytest.mark.parametrize("freeze_images", [True, False])
def test_ekf_train_filter_step(freeze_images):
    T, N, sd = 6, 32, 3
    states, obs, controls = _obs(N, sd, seed=16, T=T + 1)

    def make(src=M):
        m = fill_parameters(src.DoorCrossmodalKalmanFilter(), seed=17)
        for f in m.filter_models:
            for p in f.dynamics_model.parameters():
                p.requires_grad_(False)
        if freeze_images:
            for n, p in m.named_parameters():
                if "observation_image_layers" in n:
                    p.requires_grad_(False)
        return m

    def run(m, dev, dt):
        m.train()
        cov = (torch.eye(sd, dtype=dt) * 0.1)[None].expand(N, sd, sd).to(dev).contiguous()
        m.initialize_beliefs(mean=states[0].to(dev, dt), covariance=cov)
        est = m.forward_loop(observations={k: v[1:].to(dev, dt) for k, v in obs.items()},
                             controls=controls[1:].to(dev, dt))
        return torch.mean((est - states[1:].to(dev, dt)) ** 2)

    compare(make, run, make_ref=lambda: make(port))


@pytest.mark.gpu
def test_pf_train_filter_step():
    from oracle.noise import RecordedNoise
    from util import ReplayNoise, draw_noise

    T, N, sd, Mp = 5, 16, 2, 30
    states, obs, controls = _obs(N, sd, seed=18, T=T + 1)
    init, eps, _ = draw_noise(T, N, Mp, sd, seed=20)

    def make(src=M):
        m = fill_parameters(src.PushCrossmodalParticleFilter(), seed=19)
        for p in m.dynamics_model.parameters():
            p.requires_grad_(False)
        return m

    def run(m, dev, dt):
        m.train()
        # the same draws for all three runs (train mode: 30 particles, no resampling)
        m.noise = (ReplayNoise if dev == DEV else RecordedNoise)(init_eps=init, process_eps=list(eps), uniforms=[])
        cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(dev, dt).contiguous()
        m.initialize_beliefs(mean=states[0].to(dev, dt), covariance=cov)
        est = m.forward_loop(observations={k: v[1:].to(dev, dt) for k, v in obs.items()},
                             controls=controls[1:].to(dev, dt))
        return torch.mean((est - states[1:].to(dev, dt)) ** 2)

    # both fp32 steps evaluate the particle heads with split-bf16 operands (bf16x3), the float64 port does not: a last-bit
    # difference of a head input flips the odd ReLU of the odd particle (DESIGN.md section 9), an O(1) change of that
    # particle's contribution which either fp32 step may or may not take; the floor bounds it by 1e-3 of the largest
    # gradient, as tests/test_training_glue.py does
    compare(make, run, make_ref=lambda: make(port), floor=1e-3)
