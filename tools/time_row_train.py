"""Times training steps whose per-trajectory MLP stacks run through the row-program training kernels
(training.FusedRowProgram: mmf_row_mlp_train_fwd / _bwd / _weight_grads) against the same models with the modules'
``fused_train`` flag off (torch modules under autograd), alternating the two in one process.

Phases: train_virtual_sensor (DoorVirtualSensorModel, {pos, sensors} and {image}) and train_particle_filter_measurement
(PushMeasurementModel, proprioceptive and image head) at batch 32 and 4096; an EKF train_filter step of
DoorCrossmodalKalmanFilter (T = 15, frozen dynamics) at N = 32 / 256 / 4096 with the image encoders trainable and
frozen; the three kernels alone at 61,440 rows (the virtual-sensor program of all three modalities).  Every step is
forward + backward + buddy.minimize, CUDA events, median of --steps after --warmup; launches per step are counted with
torch.profiler (CUDA kernels) in a separate run.  Usage: python tools/time_row_train.py [--steps 20] [--warmup 5]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

from multimodalfilter_b200 import ops
from multimodalfilter_b200.crossmodal import models as M
from multimodalfilter_b200.fannypack.utils import Buddy
from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=5)
args = ap.parse_args()

dev = torch.device("cuda:0")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],  # read only
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"device: {gpu[0]}  (name, power limit); median of {args.steps} steps after {args.warmup} warm-up")


def set_row_flag(model, on):
    for m in model.modules():
        if isinstance(m, M._Encoders):
            m.fused_train = on


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def launches(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return len([e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA])


def compare(label, make, loss_fn):
    """make() -> model; loss_fn(model) -> loss.  Alternates the fused and the flag-off model."""
    runs = {}
    for on in (True, False):
        model = make().to(dev).train()
        set_row_flag(model, on)
        buddy = Buddy(f"time_row_{label}_{on}".replace(" ", "_"), model, device=str(dev))
        runs[on] = (model, buddy)
    times = {True: [], False: []}
    for i in range(args.warmup + args.steps):
        for on in (True, False):
            model, buddy = runs[on]
            t = timed(lambda: buddy.minimize(loss_fn(model), optimizer_name="train"))
            if i >= args.warmup:
                times[on].append(t)
    n = {on: launches(lambda: runs[on][1].minimize(loss_fn(runs[on][0]), optimizer_name="train")) for on in (True, False)}
    f, g = statistics.median(times[True]), statistics.median(times[False])
    print(f"{label:58s} fused {f:8.3f} ms ({n[True]:4d} launches)   torch {g:8.3f} ms ({n[False]:4d} launches)"
          f"   torch / fused {g / f:5.2f}")
    sys.stdout.flush()


def obs_batch(N, sd, T=1, seed=2):
    states, obs, controls = synthetic_trajectories(T, N, sd, seed=seed)
    return states.to(dev), {k: v.to(dev) for k, v in obs.items()}, controls.to(dev)


for B in (32, 4096):
    states, obs, _ = obs_batch(B, 3)
    o0, s0 = {k: v[0] for k, v in obs.items()}, states[0]
    for mods in ({"pos", "sensors"}, {"image"}):
        compare(f"train_virtual_sensor Door {sorted(mods)} B={B}",
                lambda: fill_parameters(M.DoorVirtualSensorModel(modalities=mods), seed=1),
                lambda m: F.mse_loss(m(observations=o0)[0], s0))
    states, obs, _ = obs_batch(B, 2)
    o0, x0 = {k: v[0] for k, v in obs.items()}, states[0][:, None, :]
    target = torch.randn(B, device=dev)
    for mods in ({"pos", "sensors"}, {"image"}):
        compare(f"train_particle_filter_measurement Push {sorted(mods)} B={B}",
                lambda: fill_parameters(M.PushMeasurementModel(modalities=mods), seed=1),
                lambda m: F.mse_loss(m(states=x0, observations=o0)[:, 0], target))

T = 15
for N in (32, 256, 4096):
    states, obs, controls = obs_batch(N, 3, T=T + 1)
    cov = (torch.eye(3, device=dev) * 0.1)[None].expand(N, 3, 3).contiguous()
    for frozen in (False, True):
        def make():
            m = fill_parameters(M.DoorCrossmodalKalmanFilter(), seed=1)
            for f in m.filter_models:
                for p in f.dynamics_model.parameters():
                    p.requires_grad_(False)
            for n, p in m.named_parameters():
                if frozen and "observation_image_layers" in n:
                    p.requires_grad_(False)
            return m

        def loss(m):
            m.initialize_beliefs(mean=states[0], covariance=cov)
            est = m.forward_loop(observations={k: v[1:] for k, v in obs.items()}, controls=controls[1:])
            return torch.mean((est - states[1:]) ** 2)

        compare(f"EKF train_filter DoorCrossmodalKF T={T} N={N} images {'frozen' if frozen else 'trainable'}", make, loss)

# ---- the kernels alone ---------------------------------------------------------------------------------------------
rows = 61440
m = fill_parameters(M.DoorVirtualSensorModel(), seed=1).to(dev)
prog = m.program()
w_fwd, w_t = prog.train_weights(dev)
g = torch.Generator(device=dev).manual_seed(0)
ins = [torch.randn(rows, d, device=dev, generator=g) for d in prog.in_dims]
d_outs = [torch.randn(rows, d, device=dev, generator=g) for d in prog.out_dims]
rev = prog.reverse((True, False, False))
state = {}


def fwd():
    state["tape"] = ops.row_mlp_train_fwd(prog.ops, w_fwd, ins, prog.in_slots, prog.out_dims, prog.out_slots, prog.scratch)[1]


def bwd():
    state["delta"] = ops.row_mlp_bwd(prog.ops, w_t, state["tape"], rev.ops, d_outs, rev.dout_slots,
                                     [prog.in_dims[i] for i in rev.inputs], rev.din_slots, rev.scratch)[1]


def dw():
    ops.row_mlp_weight_grads(prog.ops, rows, state["tape"], state["delta"], prog._w_floats)


def ev():
    ops.row_mlp(prog.ops, w_fwd, ins, prog.in_slots, prog.out_dims, prog.out_slots, prog.scratch)


macs = sum(op.in_dim * op.out_dim for op in prog.ops)
tape_mb = sum(op.in_dim + op.out_dim for op in prog.ops) * rows * 4 / 1e6
for name, fn in (("row_mlp (eval)", ev), ("row_mlp_train", fwd), ("row_mlp_bwd", bwd), ("row_mlp_dw (2 kernels)", dw)):
    ts = []
    for i in range(args.warmup + args.steps):
        t = timed(fn)
        if i >= args.warmup:
            ts.append(t)
    t = statistics.median(ts)
    print(f"{name:24s} {rows} rows of DoorVirtualSensorModel (all modalities; {macs} MAC per row, tape {tape_mb:.0f} MB): "
          f"{t * 1e3:8.1f} us  = {2 * macs * rows / t / 1e9:6.2f} TFLOP/s")
