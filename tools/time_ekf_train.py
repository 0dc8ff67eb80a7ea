"""Times one train_filter step of a Kalman model (frozen dynamics, as every curriculum of the reference) on the fused EKF
training path (training.FusedEKFLoop) against the generic path (fused_train = False), alternating the two in one process.

Per N it prints: forward + backward ms and the whole step (forward, backward, buddy.minimize) in ms, CUDA events, median
of --steps after --warmup; the recursion's own share (fused: events around FusedEKFLoop's forward / backward; generic: a
separate torch.profiler run, the self CUDA time of the ops inside the recursion's step functions); kernel launches per
step (torch.profiler, CUDA kernels).  Usage: python tools/time_ekf_train.py [--model NAME] [--T 15] [--N 32 256 4096]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from multimodalfilter_b200 import training
from multimodalfilter_b200.crossmodal import models as M
from multimodalfilter_b200.fannypack.utils import Buddy
from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories
from multimodalfilter_b200.torchfilter import filters as tf_filters

ap = argparse.ArgumentParser()
ap.add_argument("--model", default="DoorCrossmodalKalmanFilter")
ap.add_argument("--T", type=int, default=15)
ap.add_argument("--N", type=int, nargs="+", default=[32, 256, 4096])
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=5)
args = ap.parse_args()

dev = torch.device("cuda:0")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],  # read only
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"device: {gpu[0]}  (name, power limit)")
cls = dict(M.MODEL_TYPES["door"], **M.MODEL_TYPES["push"])[args.model]


class _Timed(torch.autograd.Function):
    """Identity whose forward / backward record a CUDA event: brackets FusedEKFLoop's launches in the graph."""

    @staticmethod
    def forward(ctx, tag, x):
        ctx.tag = tag
        EVENTS.setdefault(tag, []).append(torch.cuda.Event(enable_timing=True))
        EVENTS[tag][-1].record()
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        EVENTS.setdefault(ctx.tag + "_bwd", []).append(torch.cuda.Event(enable_timing=True))
        EVENTS[ctx.tag + "_bwd"][-1].record()
        return None, g


EVENTS = {}
_apply = training.FusedEKFLoop.apply


def _timed_apply(plan, mean0, cov0, controls, z, r_tril):
    # z carries gradient in every model: the backward of its wrapper runs right after the EKF backward kernel
    means, covs = _apply(plan, mean0, cov0, controls, _Timed.apply("rec_begin", z), r_tril)
    return _Timed.apply("rec_fwd_end", means), covs


def setup(N, fused):
    sd = 2 if args.model.startswith("Push") else 3
    model = fill_parameters(cls(), seed=1).to(dev).train()
    for f in getattr(model, "filter_models", [model]):
        for p in f.dynamics_model.parameters():
            p.requires_grad_(False)
    model.fused_train = fused
    buddy = Buddy(f"time_ekf_{N}_{fused}", model, device=str(dev))
    states, obs, controls = synthetic_trajectories(args.T + 1, N, sd, seed=2)
    data = (states.to(dev), {k: v.to(dev) for k, v in obs.items()}, controls.to(dev))
    return model, buddy, data


def step(model, buddy, data, minimize=True):
    states, obs, controls = data
    N, sd = states.shape[1], states.shape[2]
    cov = (torch.eye(sd, device=dev) * 0.1)[None].expand(N, sd, sd).contiguous()
    model.initialize_beliefs(mean=states[0], covariance=cov)
    est = model.forward_loop(observations={k: v[1:] for k, v in obs.items()}, controls=controls[1:])
    loss = torch.mean((est - states[1:]) ** 2)
    if minimize:
        buddy.minimize(loss, optimizer_name="train")
    else:
        loss.backward()
        model.zero_grad(set_to_none=True)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def generic_recursion_profile(model, buddy, data):
    """torch.profiler run of one generic step: CUDA time of the kernels launched inside the recursion's step functions
    (user annotations wrapped around _predict_step / _update_step), and the launches of the whole step."""
    from torch.profiler import ProfilerActivity, profile, record_function

    saved = {}
    for name in ("_predict_step", "_update_step"):
        orig = getattr(tf_filters.ExtendedKalmanFilter, name)
        saved[name] = orig

        def wrap(self, *, _orig=orig, _name=name, **kw):
            with record_function("ekf_recursion"):
                return _orig(self, **kw)

        setattr(tf_filters.ExtendedKalmanFilter, name, wrap)
    try:
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            step(model, buddy, data)
            torch.cuda.synchronize()
    finally:
        for name, orig in saved.items():
            setattr(tf_filters.ExtendedKalmanFilter, name, orig)
    kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    rec = [e for e in prof.events() if e.name == "ekf_recursion"]
    # forward kernels of the recursion (the backward ones run on autograd's thread outside the annotation)
    rec_us = sum(e.device_time_total for e in rec if hasattr(e, "device_time_total"))
    return len(kernels), rec_us / 1e3


def fused_launches(model, buddy, data):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step(model, buddy, data)
        torch.cuda.synchronize()
    return len([e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA])


print(f"model {args.model}, T = {args.T}, frozen dynamics; median of {args.steps} steps after {args.warmup} warm-up")
for N in args.N:
    runs = {True: setup(N, True), False: setup(N, False)}
    fb = {True: [], False: []}
    full = {True: [], False: []}
    share = []
    training.FusedEKFLoop.apply = _timed_apply
    for i in range(args.warmup + args.steps):
        for fused in (True, False):  # alternate the two paths
            model, buddy, data = runs[fused]
            EVENTS.clear()
            t_fb = timed(lambda: step(model, buddy, data, minimize=False))
            t_full = timed(lambda: step(model, buddy, data))
            if i >= args.warmup:
                fb[fused].append(t_fb)
                full[fused].append(t_full)
                if fused:
                    e = EVENTS
                    share.append((e["rec_begin"][-1].elapsed_time(e["rec_fwd_end"][-1]),
                                  e["rec_fwd_end_bwd"][-1].elapsed_time(e["rec_begin_bwd"][-1])))
    training.FusedEKFLoop.apply = _apply
    med = statistics.median
    f_fwd, f_bwd = med([s[0] for s in share]), med([s[1] for s in share])
    n_f = fused_launches(*runs[True])
    n_g, g_rec = generic_recursion_profile(*runs[False])
    print(f"N={N:5d}  fused:   fwd+bwd {med(fb[True]):8.3f} ms  step {med(full[True]):8.3f} ms  "
          f"recursion fwd {f_fwd:.3f} ms + bwd {f_bwd:.3f} ms  launches/step {n_f}")
    print(f"N={N:5d}  generic: fwd+bwd {med(fb[False]):8.3f} ms  step {med(full[False]):8.3f} ms  "
          f"recursion fwd {g_rec:.3f} ms (profiler, device time of the step functions' kernels)  launches/step {n_g}")
    sys.stdout.flush()
