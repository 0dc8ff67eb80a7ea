"""Times the dynamics pre-training steps on the fused rollout kernels (training.FusedDynamicsRollout) against the generic
path (fused_train = False), alternating the two in one process, and the eval rollout (DynamicsModel.forward_loop without
gradient).

Per N: one train_dynamics_recurrent step (forward_loop over T steps, MSE, backward, Adam through buddy.minimize) and one
train_dynamics_single_step step (the same on one transition), CUDA events, median of --steps after --warmup; kernel
launches per step (torch.profiler, CUDA kernels, one separate step).  Eval rollout at --eval-N x --eval-T: the one-launch
kernel that computes the control rows itself, against the same kernel fed rows computed by torch beforehand, and the
generic loop.  Usage: python tools/time_dyn_train.py [--model DoorDynamicsModel] [--T 15] [--N 32 256 4096]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

from multimodalfilter_b200 import training
from multimodalfilter_b200.crossmodal import models as M
from multimodalfilter_b200.fannypack.utils import Buddy
from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories

ap = argparse.ArgumentParser()
ap.add_argument("--model", default="DoorDynamicsModel")
ap.add_argument("--T", type=int, default=15)
ap.add_argument("--N", type=int, nargs="+", default=[32, 256, 4096])
ap.add_argument("--eval-N", type=int, default=4096)
ap.add_argument("--eval-T", type=int, default=100)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=5)
args = ap.parse_args()

dev = torch.device("cuda:0")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],  # read only
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"device: {gpu[0]}  (name, power limit)")
cls = getattr(M, args.model)
med = statistics.median


def setup(N, T, fused):
    dyn = fill_parameters(cls(), seed=1).to(dev).train()
    dyn.fused_train = fused
    buddy = Buddy(f"time_dyn_{N}_{fused}", dyn, device=str(dev))
    states, _, controls = synthetic_trajectories(T + 1, N, dyn.state_dim, seed=2)
    return dyn, buddy, (states.to(dev), controls.to(dev))


def recurrent_step(dyn, buddy, data):
    """torchfilter.train.train_dynamics_recurrent's loop body."""
    states, controls = data
    pred, _ = dyn.forward_loop(initial_states=states[0], controls=controls[1:])
    buddy.minimize(F.mse_loss(pred, states[1:]), optimizer_name="recurrent")


def single_step(dyn, buddy, data):
    """torchfilter.train.train_dynamics_single_step's loop body on the first transition of every trajectory."""
    states, controls = data
    prev, nxt, u = states[0], states[1], controls[1]
    fused = training.dynamics_rollout(dyn, prev, u[None])
    pred = fused[0] if fused is not None else dyn(initial_states=prev, controls=u)[0]
    buddy.minimize(F.mse_loss(pred, nxt), optimizer_name="single")


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


print(f"model {args.model}; median of {args.steps} after {args.warmup} warm-up, the two paths alternating")
for name, body in (("recurrent", recurrent_step), ("single_step", single_step)):
    for N in args.N:
        runs = {True: setup(N, args.T, True), False: setup(N, args.T, False)}
        ms = {True: [], False: []}
        for i in range(args.warmup + args.steps):
            for fused in (True, False):
                t = timed(lambda: body(*runs[fused]))
                if i >= args.warmup:
                    ms[fused].append(t)
        n = {fused: launches(lambda: body(*runs[fused])) for fused in (True, False)}
        steps = f"T = {args.T}" if name == "recurrent" else "T = 1"
        print(f"{name:11s} N={N:5d} {steps}: fused {med(ms[True]):8.3f} ms ({n[True]} launches)   "
              f"generic {med(ms[False]):8.3f} ms ({n[False]} launches)   speed-up {med(ms[False]) / med(ms[True]):.1f}x")
        sys.stdout.flush()

# ---- eval rollout ---------------------------------------------------------------------------------------------------
N, T = args.eval_N, args.eval_T
dyn, _, (states, controls) = setup(N, T, True)
generic, _, _ = setup(N, T, False)
plan = training._dynamics_plan(dyn)
spec = plan.dyns[0]
x0, u = states[0], controls[1:]


def given_rows():
    mid = spec.shared[0]
    rows = F.linear(dyn.control_layers(u.reshape(T * N, -1)), mid.weight[:, :64], mid.bias).reshape(T, N, 64)
    return plan.rollout(x0, rowbias=rows)


paths = {
    "fused, rows inside the kernel": lambda: dyn.forward_loop(initial_states=x0, controls=u),
    "fused kernel fed rows from torch": given_rows,
    "generic loop": lambda: generic.forward_loop(initial_states=x0, controls=u),
}
ms = {k: [] for k in paths}
with torch.no_grad():
    for i in range(args.warmup + args.steps):
        for k, fn in paths.items():
            t = timed(fn)
            if i >= args.warmup:
                ms[k].append(t)
    for k, fn in paths.items():
        print(f"eval rollout N={N} T={T}, {k:34s}: {med(ms[k]):8.3f} ms ({launches(fn)} launches)")
