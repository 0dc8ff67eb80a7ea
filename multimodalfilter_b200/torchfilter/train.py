"""``torchfilter.train``: the training loops the reference's helpers call
(ref: crossmodal/train_helpers.py:45-47,70-72,92-95,116-121,155-162; SURVEY.md Appendix A.7).

``train_filter`` is the BPTT step of BASELINE config C4: with a recognised particle filter in train mode and the dynamics
frozen (every curriculum of the reference, ref: scripts/push_task/train_push.py:154,213) each filter step runs the fused
training kernels (``training.FusedHeads``: mmf_pf_heads_forward_train / mmf_pf_heads_backward / mmf_pf_heads_weight_grads);
the optimiser step is ``buddy.minimize``, which all-reduces the gradients first when ``torch.distributed`` is initialised."""
import torch
import torch.nn.functional as F

from .. import training
from ..fannypack import utils as fp_utils
from ..fannypack.utils import SliceWrapper
from . import base


def _to_time_major(batch, device):
    """DataLoader batch (N, T, ...) -> device tensors (T, N, ...)."""
    batch = fp_utils.to_device(batch, device)
    return SliceWrapper(batch).map(lambda v: v.transpose(0, 1).contiguous()) if isinstance(batch, dict) \
        else batch.transpose(0, 1).contiguous()


def _loss(name_or_fn):
    if callable(name_or_fn):
        return name_or_fn
    assert name_or_fn == "mse", f"unsupported loss function {name_or_fn!r}"
    return F.mse_loss


def train_filter(buddy, filter_model, dataloader, *, initial_covariance, loss_function=F.mse_loss,
                 measurement_initialize=False, optimizer_name="train_filter_recurrent"):
    """One epoch of end-to-end BPTT (A.7).  Returns the mean loss of the epoch."""
    assert isinstance(filter_model, base.Filter)
    sd = filter_model.state_dim
    assert initial_covariance.shape == (sd, sd)
    loss_fn, total, batches = _loss(loss_function), 0.0, 0
    with buddy.log_scope(optimizer_name):
        for true_states, observations, controls in dataloader:
            true_states = _to_time_major(true_states, buddy.device)
            observations = _to_time_major(observations, buddy.device)
            controls = _to_time_major(controls, buddy.device)
            T, N = true_states.shape[:2]
            obs, ctrl = SliceWrapper(observations), SliceWrapper(controls)
            if measurement_initialize and hasattr(filter_model, "measurement_initialize_beliefs"):
                filter_model.measurement_initialize_beliefs(observations=obs[0])
            else:
                cov = initial_covariance.to(true_states.device)[None].expand(N, sd, sd).contiguous()
                mean = torch.distributions.MultivariateNormal(true_states[0], cov).sample()
                filter_model.initialize_beliefs(mean=mean, covariance=cov)
            predictions = filter_model.forward_loop(observations=obs[1:], controls=ctrl[1:])
            assert predictions.shape == (T - 1, N, sd)
            loss = loss_fn(predictions, true_states[1:])
            buddy.minimize(loss, optimizer_name=optimizer_name)
            buddy.log_scalar("Training loss", loss)
            total += float(loss.detach())
            batches += 1
    return total / max(batches, 1)


def train_dynamics_single_step(buddy, dynamics_model, dataloader, *, loss_function="mse",
                               optimizer_name="train_dynamics_single_step"):
    assert isinstance(dynamics_model, base.DynamicsModel)
    loss_fn, total, batches = _loss(loss_function), 0.0, 0
    with buddy.log_scope(optimizer_name):
        for batch in dataloader:
            prev, nxt, _observations, controls = fp_utils.to_device(batch, buddy.device)
            # recognised dynamics on CUDA: one step of the fused rollout (T = 1) and its reverse mode
            fused = training.dynamics_rollout(dynamics_model, prev, controls[None]) \
                if isinstance(controls, torch.Tensor) else None
            pred = fused[0] if fused is not None else dynamics_model(initial_states=prev, controls=controls)[0]
            loss = loss_fn(pred, nxt)
            buddy.minimize(loss, optimizer_name=optimizer_name)
            total += float(loss.detach())
            batches += 1
    return total / max(batches, 1)


def train_dynamics_recurrent(buddy, dynamics_model, dataloader, *, loss_function="mse",
                             optimizer_name="train_dynamics_recurrent"):
    assert isinstance(dynamics_model, base.DynamicsModel)
    loss_fn, total, batches = _loss(loss_function), 0.0, 0
    with buddy.log_scope(optimizer_name):
        for true_states, _observations, controls in dataloader:
            true_states = _to_time_major(true_states, buddy.device)
            controls = _to_time_major(controls, buddy.device)
            pred, _ = dynamics_model.forward_loop(initial_states=true_states[0], controls=SliceWrapper(controls)[1:])
            loss = loss_fn(pred, true_states[1:])
            buddy.minimize(loss, optimizer_name=optimizer_name)
            total += float(loss.detach())
            batches += 1
    return total / max(batches, 1)


def train_particle_filter_measurement(buddy, measurement_model, dataloader, *, loss_function=F.mse_loss,
                                      optimizer_name="train_measurement"):
    assert isinstance(measurement_model, base.ParticleFilterMeasurementModel)
    loss_fn, total, batches = _loss(loss_function), 0.0, 0
    with buddy.log_scope(optimizer_name):
        for batch in dataloader:
            noisy, observations, log_likelihoods = fp_utils.to_device(batch, buddy.device)
            pred = measurement_model(states=noisy[:, None, :], observations=observations)
            assert pred.shape == (noisy.shape[0], 1)
            loss = loss_fn(pred[:, 0], log_likelihoods.to(pred.dtype))
            buddy.minimize(loss, optimizer_name=optimizer_name)
            total += float(loss.detach())
            batches += 1
    return total / max(batches, 1)


def train_virtual_sensor(buddy, virtual_sensor_model, dataloader, *, loss_function="mse",
                         optimizer_name="train_virtual_sensor"):
    assert isinstance(virtual_sensor_model, base.VirtualSensorModel)
    loss_fn, total, batches = _loss(loss_function), 0.0, 0
    with buddy.log_scope(optimizer_name):
        for batch in dataloader:
            _prev, nxt, observations, _controls = fp_utils.to_device(batch, buddy.device)
            z, _ = virtual_sensor_model(observations=observations)
            loss = loss_fn(z, nxt)
            buddy.minimize(loss, optimizer_name=optimizer_name)
            total += float(loss.detach())
            batches += 1
    return total / max(batches, 1)
