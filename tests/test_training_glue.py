"""Training-loop glue (SURVEY.md section 8f rank 3): ``torchfilter.data`` / ``torchfilter.train`` / ``fannypack.utils.Buddy``
drop-ins.  CPU part: the reference's OWN ``crossmodal/train_helpers.py`` (imported from the checkout of the reference that
MMF_REFERENCE_DIR names, when there is one) runs unchanged on top of ``multimodalfilter_b200.install()`` for the phases
that are plain torch modules.  GPU part: ``train_e2e`` (ref: crossmodal/train_helpers.py:124-162), restated call for call
so that it runs without the reference, trains a PushCrossmodalParticleFilter through the fused BPTT kernels."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle.make_golden import REFERENCE, reference_available

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _trajectories(count, T, sd, seed=0):
    from multimodalfilter_b200.synthetic import synthetic_trajectories
    from multimodalfilter_b200.torchfilter.types import TrajectoryNumpy

    states, obs, controls = synthetic_trajectories(T, count, sd, seed=seed)
    return [TrajectoryNumpy(states[:, n].numpy(), {k: v[:, n].numpy() for k, v in obs.items()}, controls[:, n].numpy())
            for n in range(count)]


def test_datasets_shapes_and_coverage():
    from multimodalfilter_b200.torchfilter import data

    trajs = _trajectories(3, 21, 2)
    single = data.SingleStepDataset(trajectories=trajs)
    assert len(single) == 3 * 20
    prev, nxt, obs, ctrl = single[5]
    assert prev.shape == (2,) and nxt.shape == (2,) and obs["image"].shape == (32, 32) and ctrl.shape == (7,)
    assert np.array_equal(nxt, trajs[0].states[6]) and np.array_equal(ctrl, trajs[0].controls[6])
    sub = data.SubsequenceDataset(trajectories=trajs, subsequence_length=8)
    assert len(sub) == 3 * 2 * 2  # two sections from the front, two from the back (21 = 2 * 8 + 5)
    s, o, c = sub[0]
    assert s.shape == (8, 2) and o["gripper_pos"].shape == (8, 3) and c.shape == (8, 7)
    assert np.array_equal(sub[2][0], trajs[0].states[5:13])  # back-aligned sections start at T - 16
    batch = next(iter(torch.utils.data.DataLoader(sub, batch_size=4)))
    assert batch[0].shape == (4, 8, 2) and batch[1]["image"].shape == (4, 8, 32, 32)
    pfm = data.ParticleFilterMeasurementDataset(trajectories=trajs, covariance=np.identity(2) * 0.1, samples_per_pair=10)
    assert len(pfm) == 3 * 21 * 10
    noisy, o, ll = pfm[17]
    assert noisy.shape == (2,) and np.isfinite(ll)
    expected = -0.5 * np.sum((noisy - trajs[0].states[1]) ** 2) / 0.1 - np.log(2 * np.pi * 0.1)
    assert abs(ll - expected) < 1e-3
    assert pfm[17][0].tolist() == noisy.tolist()  # deterministic per index


def test_buddy_minimize_and_checkpoint(tmp_path):
    from multimodalfilter_b200.fannypack.utils import Buddy

    model = torch.nn.Sequential(torch.nn.Linear(3, 4), torch.nn.ReLU(), torch.nn.Linear(4, 1))
    buddy = Buddy("exp", model, device="cpu", checkpoint_dir=str(tmp_path))
    x, y = torch.randn(64, 3), torch.randn(64, 1)
    first = None
    for _ in range(50):
        loss = torch.mean((model(x) - y) ** 2)
        first = first if first is not None else float(loss.detach())
        with buddy.log_scope("train"):
            buddy.minimize(loss, optimizer_name="a")
            buddy.log_scalar("loss", loss)
    assert float(loss.detach()) < first and buddy.optimizer_steps == 50 and len(buddy.scalars["train/loss"]) == 50
    buddy.save_checkpoint("phase0")
    w = model[0].weight.detach().clone()
    with torch.no_grad():
        model[0].weight.zero_()
    buddy.load_checkpoint("phase0")
    assert torch.equal(model[0].weight, w)
    with torch.no_grad():
        model[2].weight.zero_()
    buddy.load_checkpoint_module("2", label="phase0")
    assert model[2].weight.abs().sum() > 0


@pytest.mark.skipif(not reference_available(), reason="MMF_REFERENCE_DIR does not name a checkout of the reference")
def test_reference_train_helpers_run_on_the_drop_in():
    """ref: crossmodal/train_helpers.py, imported unchanged: configure() + the three pre-training phases whose models are
    plain torch modules (dynamics single-step / recurrent, PF measurement, virtual sensor) on CPU."""
    code = r'''
import sys, warnings
sys.path.insert(0, %r); sys.path.insert(1, %r)
warnings.filterwarnings("ignore")
import multimodalfilter_b200 as mmf; mmf.install()
import fannypack, torch, torchfilter
sys.path.insert(2, %r)
import crossmodal
from crossmodal import train_helpers
from test_training_glue import _trajectories
torch.manual_seed(0)
model = crossmodal.push_models.PushCrossmodalParticleFilter()
buddy = fannypack.utils.Buddy("glue", model, device="cpu")
train_helpers.configure(buddy=buddy, trajectories=_trajectories(4, 12, 2), num_workers=0)
train_helpers.train_pf_dynamics_single_step(epochs=1, batch_size=8)
train_helpers.train_pf_dynamics_recurrent(subsequence_length=4, epochs=1, batch_size=4)
fannypack.utils.freeze_module(model.dynamics_model)
train_helpers.train_pf_measurement(epochs=1, batch_size=64)
steps = buddy.optimizer_steps
assert steps == 6 + 3 + 8, steps  # ceil(44 / 8) + 12 / 4 + ceil(480 / 64) optimiser steps
kf = crossmodal.door_models.DoorKalmanFilter()
buddy2 = fannypack.utils.Buddy("glue_kf", kf, device="cpu")
train_helpers.configure(buddy=buddy2, trajectories=_trajectories(3, 6, 3), num_workers=0)
train_helpers.train_virtual_sensor(epochs=1, batch_size=5)
assert buddy2.optimizer_steps == 3
print("OK")
''' % (REPO, os.path.join(REPO, "tests"), REFERENCE)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and "OK" in res.stdout, (res.stdout[-2000:], res.stderr[-3000:])


@pytest.mark.gpu
def test_train_e2e_runs_the_fused_bptt_step():
    """train_e2e restated call for call (ref: crossmodal/train_helpers.py:124-162): SubsequenceDataset -> DataLoader
    (shuffle, drop_last) -> torchfilter.train.train_filter(buddy, model, dataloader, initial_covariance=, ...), with the
    curriculum's frozen dynamics (ref: scripts/push_task/train_push.py:83-104).  The loss must go down and the fused
    training kernels must be the ones that ran."""
    import multimodalfilter_b200.fannypack as fannypack
    import multimodalfilter_b200.torchfilter as torchfilter
    from multimodalfilter_b200 import ops
    from multimodalfilter_b200.crossmodal import models as M
    from multimodalfilter_b200.synthetic import fill_parameters

    torch.manual_seed(0)
    model = fill_parameters(M.PushCrossmodalParticleFilter(), seed=3)
    buddy = fannypack.utils.Buddy("glue_e2e", model, device="cuda:0")
    fannypack.utils.freeze_module(model.dynamics_model)
    trajectories = _trajectories(32, 17, 2, seed=5)

    def train_e2e(*, subsequence_length, epochs, batch_size=32, initial_cov_scale=0.1, measurement_initialize=False,
                  optimizer_name="train_filter_recurrent"):
        model.train()
        dataloader = torch.utils.data.DataLoader(
            torchfilter.data.SubsequenceDataset(trajectories=trajectories, subsequence_length=subsequence_length),
            batch_size=batch_size, shuffle=True, num_workers=0, drop_last=True)
        initial_covariance = torch.eye(model.state_dim, device=buddy.device) * initial_cov_scale
        return [torchfilter.train.train_filter(buddy, model, dataloader, initial_covariance=initial_covariance,
                                               measurement_initialize=measurement_initialize,
                                               optimizer_name=optimizer_name) for _ in range(epochs)]

    ops.PROFILE.reset()
    losses = train_e2e(subsequence_length=16, epochs=6, batch_size=16)
    assert buddy.optimizer_steps == 6 * 4  # 32 trajectories x 2 alignments / 16 per batch
    assert ops.PROFILE.launches >= 24 * 15 * 3, "the fused BPTT kernels did not run"
    assert np.isfinite(losses).all() and losses[-1] < losses[0], losses
    assert all(p.grad is None for p in model.dynamics_model.parameters())
    assert any(p.grad is not None and p.grad.abs().sum() > 0 for n, p in model.named_parameters()
               if "observation_image_layers.0" in n), "the image-encoder CNN received no gradient"


@pytest.mark.gpu
def test_training_forward_loop_hoists_the_per_trajectory_pieces():
    """forward_loop in train mode computes encoders / weight model / the heads' observation rows once over all T * N rows
    and then runs the per-particle kernels step by step: loss and every parameter gradient must equal T calls of forward()
    (same draws) to fp32 rounding, and parameters of the encoders must receive gradients on both routes."""
    import torch
    from multimodalfilter_b200 import ops
    from multimodalfilter_b200.crossmodal import models as M
    from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories
    from util import ReplayNoise, assert_close, draw_noise

    dev, sd, N, Mp, T = "cuda:0", 2, 12, 30, 6
    init, eps, _ = draw_noise(T, N, Mp, sd, seed=51)
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=52)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(dev).contiguous()
    o = {k: v[1:].to(dev) for k, v in obs.items()}
    c = controls[1:].to(dev)
    target = states[1:].to(dev)
    results = []
    for hoisted in (False, True):
        f = fill_parameters(M.PushCrossmodalParticleFilter(), seed=53).to(dev)
        f.train()
        for p in f.dynamics_model.parameters():
            p.requires_grad_(False)  # the reference's end-to-end curricula freeze the dynamics
        f.noise = ReplayNoise(init_eps=init, process_eps=list(eps), uniforms=[])
        f.initialize_beliefs(mean=states[0].to(dev), covariance=cov)
        ops.PROFILE.reset(enabled=True)
        if hoisted:
            est = f.forward_loop(observations=o, controls=c)
        else:
            est = torch.stack([f.forward(observations={k: v[t] for k, v in o.items()}, controls=c[t]) for t in range(T)])
        loss = torch.mean((est - target) ** 2)
        loss.backward()
        kernels = ops.PROFILE.collect()["kernels"]
        ops.PROFILE.reset()
        assert kernels["pf_heads_forward_train"]["count"] == T and kernels["pf_reweight_train_bwd"]["count"] == T
        assert kernels["pf_traj_rows"]["count"] == (1 if hoisted else T)
        results.append((float(loss), {k: p.grad.detach().cpu().clone() for k, p in f.named_parameters() if p.grad is not None}))
    (l0, g0), (l1, g1) = results
    assert abs(l0 - l1) <= 1e-6 * abs(l0)
    assert set(g0) == set(g1) and len(g0) > 80 and any("observation_image_layers" in k for k in g0)
    # Same mathematics, different batching of the library GEMMs / cuDNN (12 rows per step vs 72 at once): the per-trajectory
    # rows differ in the last bit, which flips the odd ReLU of the odd particle (an O(1) change of that particle's
    # contribution, DESIGN.md section 9) and re-orders the CNN's heavily cancelling weight-gradient sums.  The check is
    # therefore per tensor: direction and magnitude; a missing or doubled contribution would show up as O(1).
    big = max(float(g.norm()) for g in g0.values())
    for k in g0:
        a, b = g1[k].double().reshape(-1), g0[k].double().reshape(-1)
        rel = float((a - b).norm() / max(float(b.norm()), 1e-3 * big))
        cos = float(torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-30)) if float(b.norm()) > 1e-3 * big else 1.0
        assert rel <= 2e-2 and cos >= 0.999, f"{k}: relative L2 {rel:.2e}, cosine {cos:.5f}"
