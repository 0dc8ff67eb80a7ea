"""Drop-in counterparts of the reference's ``crossmodal`` model classes (same class names,
constructor arguments, attributes and ``state_dict`` keys, so reference checkpoints load and the
reference's scripts run), wired to the CUDA kernels.

The per-particle and per-trajectory arithmetic is NOT evaluated by these modules on the fused
path: they are parameter containers whose weights ``fused.py`` packs for the kernels.  Their
``forward`` methods are the generic (torch-on-GPU) path used when gradients are required.

ref: crossmodal/base_models/*.py, crossmodal/push_models/*.py, crossmodal/door_models/*.py
"""
import abc
from typing import List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from .. import fused, ops, training
from ..encoders import ImageEncoder
from ..fannypack.nn import resblocks
from ..fannypack.utils import SliceWrapper
from ..torchfilter import base as tf_base
from ..torchfilter import filters as tf_filters

UNITS = 64
DIMS = {"control": 7, "pos": 3, "sensors": 7}  # ref: crossmodal/push_models/layers.py:5-8


# ---- building blocks ---------------------------------------------------------------------------------
def _mlp_encoder(n_in: int, units: int) -> nn.Sequential:
    # ref: crossmodal/push_models/layers.py:11-40,107-136
    return nn.Sequential(nn.Linear(n_in, units), nn.ReLU(inplace=True), resblocks.Linear(units))


class _SpanningMeans(nn.Module):
    # ref: crossmodal/push_models/layers.py:43-65
    def __init__(self, rows, cols, reduce_size=1):
        super().__init__()
        self.pool_h = nn.Sequential(nn.AvgPool2d((rows, reduce_size)), nn.Flatten())
        self.pool_w = nn.Sequential(nn.AvgPool2d((reduce_size, cols)), nn.Flatten())

    def forward(self, x):
        return torch.cat((self.pool_h(x), self.pool_w(x)), dim=-1)


def _image_encoder(units: int, spanning_avg_pool: bool = False) -> nn.Sequential:
    # ref: crossmodal/push_models/layers.py:68-104, crossmodal/door_models/layers.py:43-63
    layers = [
        nn.Conv2d(1, 32, 5, padding=2), nn.ReLU(inplace=True),
        resblocks.Conv2d(32, kernel_size=3),
        nn.Conv2d(32, 16, 3, padding=1), nn.ReLU(inplace=True),
    ]
    if spanning_avg_pool:
        layers += [nn.Conv2d(16, 2, 3, padding=1), _SpanningMeans(32, 32, reduce_size=2), nn.Linear(64, units)]
    else:
        layers += [nn.Conv2d(16, 8, 3, padding=1), nn.Flatten(), nn.Linear(8 * 32 * 32, units)]
    layers += [nn.ReLU(inplace=True), resblocks.Linear(units)]
    return ImageEncoder(*layers)


class _Encoders(nn.Module):
    """Holds ``observation_{image,pos,sensors}_layers`` for a modality subset."""

    def _make_encoders(self, modalities, units, spanning_avg_pool=False):
        valid = {"image", "pos", "sensors"}
        assert len(valid | set(modalities)) == 3, "Received invalid modality"
        assert len(modalities) > 0, "Received empty modality list"
        self.modalities = set(modalities)
        if "image" in self.modalities:
            self.observation_image_layers = _image_encoder(units, spanning_avg_pool)
        if "pos" in self.modalities:
            self.observation_pos_layers = _mlp_encoder(DIMS["pos"], units)
        if "sensors" in self.modalities:
            self.observation_sensors_layers = _mlp_encoder(DIMS["sensors"], units)

    def encode(self, observations):
        parts = []
        for mod, attr in fused.OBS_ORDER:
            if mod in self.modalities:
                x = observations[fused.OBS_KEY[mod]]
                parts.append(getattr(self, attr)(x[:, None] if mod == "image" else x))
        return torch.cat(parts, dim=1)

    def _encoder_list(self):
        return [(mod, getattr(self, attr)) for mod, attr in fused.OBS_ORDER if mod in self.modalities]

    def encoded_program(self, key, tails, units=UNITS):
        """One ``mmf_row_mlp`` program for "encode the non-image modalities, concatenate, run the tail stacks":
        ``tails`` = list of (nn.Sequential, column offset into the first tail's output or None for the concatenated
        features, input width); each tail's result is an output.  Image features are an input (CNN trunk kernel +
        Linear tail run as the module).  Cached per module; None when a stack is not fusable."""
        def build():
            prog = fused.RowProgram()
            encs = self._encoder_list()
            base = prog.alloc(units * len(encs), fresh=True)  # holds an input (the image features): never a recycled slot
            for i, (mod, enc) in enumerate(encs):
                if mod == "image":
                    prog.input(units, slot=base + units * i)
                else:
                    src = prog.input(enc[0].in_features)
                    prog.sequential(enc, src, enc[0].in_features, dst=base + units * i)
                    prog.release(src, enc[0].in_features)  # the raw input is dead once its encoder has run
            first = None
            for seq, offset, width in tails:
                src = base if offset is None else first + offset
                slot, dim = prog.sequential(seq, src, width)
                if offset is None and src == base:
                    prog.release(base, units * len(encs))  # the concatenated features: consumed by the first tail only
                first = slot if first is None else first
                if offset is not None or len(tails) == 1:
                    prog.output(slot, dim)
            return prog

        return fused.cached_program(self, key, build)

    def program_inputs(self, observations):
        """Inputs of ``encoded_program`` in its order, or None when the fused launch does not apply."""
        encs = self._encoder_list()
        raw = [observations[fused.OBS_KEY[mod]] for mod, _ in encs if mod != "image"]
        if not fused.row_program_ok(*raw) or ("image" in self.modalities and not observations["image"].is_cuda):
            return None
        return [enc(observations["image"][:, None]) if mod == "image" else observations[fused.OBS_KEY[mod]]
                for mod, enc in encs]


def _blackout_rows(observations):
    img = observations["image"]
    return img.reshape(img.shape[0], -1).abs().sum(dim=1) < 1e-8  # ref: push_models/crossmodal_pf.py:97-101


class _EnabledModels:
    """``enabled_models`` with the reference's validation; scripts also assign ``_enabled_models``
    directly (ref: scripts/push_task/train_push.py:157,165,176), so it is read at call time."""

    @property
    def enabled_models(self) -> List[bool]:
        return self._enabled_models

    @enabled_models.setter
    def enabled_models(self, flags: List[bool]) -> None:
        assert isinstance(flags, list)
        assert len(flags) == len(self._enabled_models)
        for f in flags:
            assert type(f) == bool
        self._enabled_models = flags


# ---- dynamics (R3) -------------------------------------------------------------------------------------
class _Dynamics(tf_base.DynamicsModel):
    _mmf_fusable = True
    _STATE_DIM = None
    _NOISE = None  # ("tril" | "diag", variances, divisor)

    def __init__(self, units=UNITS):
        super().__init__(state_dim=self._STATE_DIM)
        kind, variances, divisor = self._NOISE
        sigma = torch.sqrt(torch.tensor(variances, dtype=torch.float32)) / divisor
        if kind == "tril":
            self.Q_scale_tril = nn.Parameter(torch.diag(sigma), requires_grad=False)
        else:
            self.Q_scale_tril_diag = nn.Parameter(sigma, requires_grad=False)
        self.state_layers = _mlp_encoder(self.state_dim, units)
        self.control_layers = _mlp_encoder(DIMS["control"], units)
        self.shared_layers = nn.Sequential(
            nn.Linear(2 * units, units),
            resblocks.Linear(units), resblocks.Linear(units), resblocks.Linear(units),
            nn.Linear(units, self.state_dim + 1),
        )
        self.units = units

    def scale_tril(self):
        return self.Q_scale_tril if hasattr(self, "Q_scale_tril") else torch.diag(self.Q_scale_tril_diag)

    def forward(self, *, initial_states, controls):
        N, sd = initial_states.shape[:2]
        assert sd == self.state_dim
        h = self.shared_layers(torch.cat((self.control_layers(controls), self.state_layers(initial_states)), dim=-1))
        nxt = initial_states + h[..., :sd] * torch.sigmoid(h[..., sd:])
        return nxt, self.scale_tril()[None].expand(N, sd, sd)


class PushDynamicsModel(_Dynamics):  # ref: crossmodal/push_models/dynamics.py:10-64
    _STATE_DIM, _NOISE = 2, ("tril", [0.02, 0.02], 1.0)


class DoorDynamicsModel(_Dynamics):  # ref: crossmodal/door_models/dynamics.py:11-67
    _STATE_DIM, _NOISE = 3, ("tril", [0.05, 0.01, 0.01], 1.0)


class DoorDynamicsModelBrent(_Dynamics):  # ref: crossmodal/door_models/dynamics.py:76-134
    _STATE_DIM, _NOISE = 3, ("diag", [0.05, 0.01, 0.01], 8.0)


# ---- particle-filter measurement side (R4, R5) ------------------------------------------------------------
class _Head(tf_base.ParticleFilterMeasurementModel, _Encoders):
    _mmf_fusable = True
    _STATE_DIM = None

    def __init__(self, units: int = UNITS, modalities=frozenset({"image", "pos", "sensors"})):
        super().__init__(state_dim=self._STATE_DIM)
        self._make_encoders(modalities, units)
        self.state_layers = _mlp_encoder(self.state_dim, units)
        self.shared_layers = nn.Sequential(
            nn.Linear(units * (1 + len(self.modalities)), units), nn.ReLU(inplace=True),
            resblocks.Linear(units), resblocks.Linear(units),
            nn.Linear(units, 1),
        )
        self.units = units

    def forward(self, *, states, observations):
        assert type(observations) == dict
        assert states.dim() == 3 and states.shape[2] == self.state_dim
        N, M, _ = states.shape
        f_obs = self.encode(observations)
        merged = torch.cat((f_obs[:, None, :].expand(N, M, f_obs.shape[1]), self.state_layers(states)), dim=2)
        return self.shared_layers(merged)[..., 0]


class PushMeasurementModel(_Head):  # ref: crossmodal/push_models/pf.py:30-109
    _STATE_DIM = 2


class DoorMeasurementModel(_Head):  # ref: crossmodal/door_models/pf.py:28-107
    _STATE_DIM = 3


class CrossmodalWeightModel(nn.Module, abc.ABC):  # ref: crossmodal/base_models/crossmodal_pf.py:11-30
    def __init__(self, modality_count: int):
        super().__init__()
        self.modality_count = modality_count

    @abc.abstractmethod
    def forward(self, *, observations) -> torch.Tensor:
        ...


class CrossmodalParticleFilterMeasurementModel(tf_base.ParticleFilterMeasurementModel, _EnabledModels):
    """ref: crossmodal/base_models/crossmodal_pf.py:33-141.  On the fused path the K heads and this
    fusion run inside ``mmf_pf_predict_measure``; this ``forward`` serves the gradient path, with the
    fusion itself in ``mmf_fuse_loglik`` when no gradient is needed."""

    _mmf_fusable = True

    def __init__(self, *, measurement_models, crossmodal_weight_model: Optional[CrossmodalWeightModel], state_dim: int):
        super().__init__(state_dim=state_dim)
        self.measurement_models = nn.ModuleList(measurement_models)
        self.crossmodal_weight_model = crossmodal_weight_model
        self._enabled_models = [True] * len(self.measurement_models)

    def forward(self, *, states, observations):
        N, M, _ = states.shape
        on = self._enabled_models
        ll = torch.stack(
            [m(states=states, observations=observations) for i, m in enumerate(self.measurement_models) if on[i]], dim=2
        )
        assert ll.shape == (N, M, int(np.sum(on)))
        w = None
        if self.crossmodal_weight_model is not None:
            w = self.crossmodal_weight_model(observations=observations)[:, on]
            assert w.shape == (N, int(np.sum(on)))
        if torch.is_grad_enabled() and (ll.requires_grad or (w is not None and w.requires_grad)):
            return torch.logsumexp(ll if w is None else w[:, None, :] + ll, dim=2)
        return ops.fuse_loglik(ll, None if w is None else w.contiguous())


class _PFWeights(CrossmodalWeightModel, _Encoders):
    _RES = 1

    def __init__(self, know_image_blackout: bool, units: int = UNITS):
        super().__init__(modality_count=2)
        self.know_image_blackout = know_image_blackout
        self._make_encoders({"image", "pos", "sensors"}, units)
        self.fusion_layers = nn.Sequential(
            nn.Linear(3 * units, units), nn.ReLU(inplace=True),
            *[resblocks.Linear(units) for _ in range(self._RES)],
            nn.Linear(units, 2),
        )

    def forward(self, *, observations):
        ins = self.program_inputs(observations)
        prog = self.encoded_program("weights", [(self.fusion_layers, None, 3 * UNITS)]) if ins is not None else None
        out = prog.run(ins)[0] if prog is not None else self.fusion_layers(self.encode(observations))
        assert out.shape == (observations["gripper_pos"].shape[0], self.modality_count)
        if self.know_image_blackout:
            out[_blackout_rows(observations), 0] -= np.inf  # quirk Q3
        return out


class PushCrossmodalWeightModel(_PFWeights):  # ref: crossmodal/push_models/crossmodal_pf.py:52-104
    _RES = 1


class DoorCrossmodalWeightModel(_PFWeights):  # ref: crossmodal/door_models/crossmodal_pf.py:52-106
    _RES = 3


class _TaskPF(tf_filters.ParticleFilter):
    def train(self, mode: bool = True):
        self.num_particles = 30 if mode else 300  # quirk Q8, ref: crossmodal/push_models/pf.py:24-27
        return super().train(mode)


def _make_pf_classes(prefix, dyn_cls, head_cls, weight_cls, sd):
    def two_heads():
        return [head_cls(modalities={"image"}), head_cls(modalities={"pos", "sensors"})]

    def plain_init(self):
        tf_filters.ParticleFilter.__init__(self, dynamics_model=dyn_cls(), measurement_model=head_cls(), num_particles=30)

    def crossmodal_init(self, know_image_blackout: bool = False):
        tf_filters.ParticleFilter.__init__(
            self, dynamics_model=dyn_cls(),
            measurement_model=CrossmodalParticleFilterMeasurementModel(
                measurement_models=two_heads(),
                crossmodal_weight_model=weight_cls(know_image_blackout=know_image_blackout), state_dim=sd),
            num_particles=30,
        )

    def unimodal_init(self):
        tf_filters.ParticleFilter.__init__(
            self, dynamics_model=dyn_cls(),
            measurement_model=CrossmodalParticleFilterMeasurementModel(
                measurement_models=two_heads(), crossmodal_weight_model=None, state_dim=sd),
            num_particles=30,
        )

    plain = type(prefix + "ParticleFilter", (_TaskPF,), {"__init__": plain_init})
    cross = type(prefix + "CrossmodalParticleFilter", (_TaskPF,), {"__init__": crossmodal_init})
    seq5 = type(prefix + "CrossmodalParticleFilterSeq5", (cross,),
                {"__init__": lambda self: crossmodal_init(self, know_image_blackout=True)})
    uni = type(prefix + "UnimodalParticleFilter", (_TaskPF,), {"__init__": unimodal_init})
    return plain, cross, seq5, uni


(PushParticleFilter, PushCrossmodalParticleFilter, PushCrossmodalParticleFilterSeq5,
 PushUnimodalParticleFilter) = _make_pf_classes("Push", PushDynamicsModel, PushMeasurementModel, PushCrossmodalWeightModel, 2)
(DoorParticleFilter, DoorCrossmodalParticleFilter, DoorCrossmodalParticleFilterSeq5,
 DoorUnimodalParticleFilter) = _make_pf_classes("Door", DoorDynamicsModelBrent, DoorMeasurementModel, DoorCrossmodalWeightModel, 3)


# ---- Kalman side (R8-R12) ----------------------------------------------------------------------------------
class _VirtualSensor(tf_base.VirtualSensorModel, _Encoders):
    _STATE_DIM = None
    _SPANNING = False

    def __init__(self, units: int = UNITS, modalities=frozenset({"image", "pos", "sensors"}), add_R_noise: float = 1e-6,
                 noise_R_tril: torch.Tensor = None):
        super().__init__(state_dim=self._STATE_DIM)
        sd = self.state_dim
        self.noise_R_tril = noise_R_tril
        self._make_encoders(modalities, units, spanning_avg_pool=self._SPANNING)
        self.shared_layers = nn.Sequential(
            nn.Linear(units * len(self.modalities), 2 * units), nn.ReLU(inplace=True),
            resblocks.Linear(2 * units), resblocks.Linear(2 * units),
        )
        self.r_layer = nn.Sequential(nn.Linear(units, sd), nn.ReLU(inplace=True), resblocks.Linear(sd), nn.Linear(sd, sd))
        self.z_layer = nn.Sequential(nn.Linear(units, sd), nn.ReLU(inplace=True), resblocks.Linear(sd), nn.Linear(sd, sd))
        self.units = units
        self.add_R_noise = torch.ones(sd) * add_R_noise

    def forward(self, *, observations):
        # R9, ref: crossmodal/door_models/kf.py:81-126
        assert type(observations) == dict
        ins = self.program_inputs(observations) if self.noise_R_tril is None else None
        prog = None
        if ins is not None:  # encoders + shared stack + both heads in one launch (mmf_row_mlp)
            prog = self.encoded_program("sensor", [(self.shared_layers, None, self.units * len(self.modalities)),
                                                   (self.z_layer, 0, self.units), (self.r_layer, self.units, self.units)])
        if prog is not None:
            z, lt_hat = prog.run(ins)
        else:
            h = self.shared_layers(self.encode(observations))
            z = self.z_layer(h[:, : self.units].clone())
            lt_hat = self.r_layer(h[:, self.units :].clone()) if self.noise_R_tril is None else self.noise_R_tril
        R = torch.diag_embed(lt_hat) ** 2
        if self.add_R_noise[0] > 0:
            R = R + torch.diag(self.add_R_noise).to(R.device)
        return z, torch.sqrt(R)


class PushVirtualSensorModel(_VirtualSensor):  # ref: crossmodal/push_models/kf.py:31-128
    _STATE_DIM, _SPANNING = 2, True


class DoorVirtualSensorModel(_VirtualSensor):  # ref: crossmodal/door_models/kf.py:31-126
    _STATE_DIM = 3


def _make_kf_class(name, dyn_cls, sensor_cls):
    def init(self, dynamics_model=None, virtual_sensor_model=None):
        if dynamics_model is None and virtual_sensor_model is None:
            dynamics_model, virtual_sensor_model = dyn_cls(), sensor_cls()
        tf_filters.VirtualSensorExtendedKalmanFilter.__init__(
            self, dynamics_model=dynamics_model, virtual_sensor_model=virtual_sensor_model)

    return type(name, (tf_filters.VirtualSensorExtendedKalmanFilter,), {"__init__": init})


PushKalmanFilter = _make_kf_class("PushKalmanFilter", PushDynamicsModel, PushVirtualSensorModel)
DoorKalmanFilter = _make_kf_class("DoorKalmanFilter", DoorDynamicsModel, DoorVirtualSensorModel)


def weighted_average(predictions, weights):  # ref: crossmodal/base_models/utility.py:4-11
    assert predictions.shape == weights.shape
    weights = weights / (torch.sum(weights, dim=0) + 1e-9)
    return torch.sum(weights * predictions, dim=0)


class CrossmodalKalmanFilterWeightModel(nn.Module, abc.ABC):  # ref: base_models/crossmodal_kf.py:13-36
    def __init__(self, modality_count: int, state_dim: int):
        super().__init__()
        self.modality_count = modality_count
        self.state_dim = state_dim

    @abc.abstractmethod
    def forward(self, *, observations) -> torch.Tensor:
        ...


class _KFWeights(CrossmodalKalmanFilterWeightModel, _Encoders):
    """ref: crossmodal/door_models/crossmodal_kf.py:101-167."""

    def __init__(self, units: int = UNITS, state_dim: int = 2, know_image_blackout=False):
        super().__init__(modality_count=2, state_dim=state_dim)
        self._make_encoders({"image", "pos", "sensors"}, units)
        self.weighting_type = "sigmoid"
        self.fusion_layers = nn.Sequential(
            nn.Linear(3 * units, units), nn.ReLU(inplace=True), resblocks.Linear(units),
            nn.Linear(units, 2 * state_dim), nn.Sigmoid(),
        )
        self.know_image_blackout = know_image_blackout

    def raw(self, observations):
        ins = self.program_inputs(observations)
        prog = self.encoded_program("weights", [(self.fusion_layers, None, 3 * UNITS)]) if ins is not None else None
        if prog is not None:  # encoders + fusion stack + sigmoid in one launch
            return prog.run(ins)[0]
        return self.fusion_layers(self.encode(observations))

    @staticmethod
    def shape_weights(out, K, N, sd):
        beta = out.reshape(K, N, sd)  # quirk Q5: row-major reinterpretation, mixes trajectories
        return beta / (beta.sum(dim=0) + 1e-9)

    def forward(self, *, observations):
        N = observations["gripper_pos"].shape[0]
        out = self.raw(observations)
        assert out.shape == (N, self.modality_count * self.state_dim)
        return self.shape_weights(out, self.modality_count, N, self.state_dim)

    def forward_sequence(self, observations, T, N):
        """(T, K, N, sd): the per-step reshape applied to a time-batched encoder pass."""
        chunks = fused.batched_over_time(self.raw, observations, T, N)
        out = torch.cat(chunks).reshape(T, self.modality_count, N, self.state_dim)
        return out / (out.sum(dim=1, keepdim=True) + 1e-9)


class PushCrossmodalKalmanFilterWeightModel(_KFWeights):
    pass


class DoorCrossmodalKalmanFilterWeightModel(_KFWeights):
    pass


def _mask_weights(flags, N, sd, device):  # ref: base_models/crossmodal_kf.py:124-131
    w = torch.tensor(flags, dtype=torch.float32, device=device)
    return w[:, None, None].repeat(1, N, sd)


def _fuse_kernel_ok(*tensors) -> bool:
    """mmf_kf_fuse_measurements serves inference on CUDA fp32 tensors; autograd keeps the torch expressions."""
    return not torch.is_grad_enabled() and all(t.is_cuda and t.dtype == torch.float32 for t in tensors)


def _measurement_level(states, trils, weights):  # ref: base_models/crossmodal_kf.py:219-235,337-354
    covs = trils @ trils.transpose(-1, -2)
    mult = torch.prod(torch.prod(weights, dim=-1), dim=0)[:, None, None]
    return weighted_average(states, weights), mult * covs.sum(dim=0)


class _MultiFilter(tf_base.Filter, _EnabledModels):
    """Shared machinery of Crossmodal/Unimodal KalmanFilter: K independent EKFs advanced by ONE
    ``mmf_ekf_loop_fwd`` launch (no posterior feedback, quirk Q6), then a fusion kernel."""

    def __init__(self, *, filter_models, state_dim: int):
        super().__init__(state_dim=state_dim)
        self.filter_models = nn.ModuleList(filter_models)
        self._enabled_models = [True] * len(self.filter_models)
        self.weighted_covariances = None
        self.fused_train = True  # training with frozen dynamics: the F filters' recursion and its backward as one kernel each

    @property
    def fused_train(self):
        return self.__dict__.get("_mmf_fused_train", True)

    @fused_train.setter
    def fused_train(self, on):
        # the member filters follow, so that the step-by-step path (forward) agrees with forward_loop
        self.__dict__["_mmf_fused_train"] = bool(on)
        for f in self.filter_models:
            f.fused_train = bool(on)

    @property
    def state_covariance_estimate(self):
        return self.weighted_covariances

    def initialize_beliefs(self, *, mean, covariance):
        N = mean.shape[0]
        assert mean.shape == (N, self.state_dim)
        assert covariance.shape == (N, self.state_dim, self.state_dim)
        for f in self.filter_models:
            f.initialize_beliefs(mean=mean, covariance=covariance)

    def _enabled_filters(self):
        return [f for f, on in zip(self.filter_models, self._enabled_models) if on]

    def _plan(self, filters):
        key = tuple(f.dynamics_model for f in filters)  # the modules themselves, compared by identity
        cached = self.__dict__.get("_mmf_plan")
        if cached is None or len(cached[0]) != len(key) or any(a is not b for a, b in zip(cached[0], key)):
            ok = all(isinstance(f, tf_filters.VirtualSensorExtendedKalmanFilter) for f in filters)
            cached = (key, fused.EKFPlan.build(filters) if ok else None)
            self.__dict__["_mmf_plan"] = cached
        return cached[1]

    def _fusable(self, filters, controls):
        return (
            isinstance(controls, torch.Tensor) and controls.is_cuda and self._plan(filters) is not None
            and not tf_filters._needs_grad(self, *[f._belief_mean for f in filters])
            and all(f._initialized for f in filters)
        )

    def _advance(self, filters, controls, z, r_tril):
        """controls (T,N,cd), z / r_tril (F,T,N,...) -> posterior means (F,T,N,sd), covs."""
        mean0 = torch.stack([f._belief_mean.detach() for f in filters])
        cov0 = torch.stack([f._belief_covariance.detach() for f in filters])
        means, covs = self._plan(filters).loop(mean0, cov0, controls, z, r_tril)
        for i, f in enumerate(filters):
            f._belief_mean, f._belief_covariance = means[i, -1], covs[i, -1]
        return means, covs

    def _train_fused(self, filters, controls, observations):
        return all(f._initialized for f in filters) and training.fused_ekf_train_applicable(
            self, filters, self._plan(filters), controls, observations,
            [t for f in filters for t in (f._belief_mean, f._belief_covariance)])

    def _advance_train(self, filters, controls, z, r_tril):
        """``_advance`` with autograd (``training.FusedEKFLoop``): the new beliefs keep their ``grad_fn``."""
        mean0 = torch.stack([f._belief_mean for f in filters])
        cov0 = torch.stack([f._belief_covariance for f in filters])
        means, covs = training.FusedEKFLoop.apply(self._plan(filters), mean0, cov0, controls, z, r_tril)
        for i, f in enumerate(filters):
            f._belief_mean, f._belief_covariance = means[i, -1], covs[i, -1]
        return means, covs

    def _sense_sequence_train(self, filters, observations, T, N):
        zr = [f.sense_sequence(observations, T, N, grad=True) for f in filters]
        return torch.stack([a[0] for a in zr]), torch.stack([a[1] for a in zr])

    def calculate_unimodal_states(self, observations, controls):
        filters = self._enabled_filters()
        if self._train_fused(filters, controls, observations):
            zr = [f.virtual_sensor_model(observations=observations) for f in filters]
            z = torch.stack([a[0] for a in zr])[:, None]
            r = torch.stack([a[1] for a in zr])[:, None]
            means, covs = self._advance_train(filters, controls[None], z, r)
            return means[:, 0], covs[:, 0]
        if self._fusable(filters, controls):
            zr = [f.virtual_sensor_model(observations=observations) for f in filters]
            z = torch.stack([a[0].detach() for a in zr])[:, None]
            r = torch.stack([a[1].detach() for a in zr])[:, None]
            means, covs = self._advance(filters, controls[None], z, r)
            return means[:, 0], covs[:, 0]
        states = torch.stack([f(observations=observations, controls=controls) for f in filters])
        covs = torch.stack([f._belief_covariance for f in filters])
        return states, covs


class CrossmodalKalmanFilter(_MultiFilter):
    """ref: crossmodal/base_models/crossmodal_kf.py:39-240."""

    def __init__(self, *, filter_models, crossmodal_weight_model: CrossmodalKalmanFilterWeightModel, state_dim: int):
        super().__init__(filter_models=filter_models, state_dim=state_dim)
        self.crossmodal_weight_model = crossmodal_weight_model

    def calculate_weighted_states(self, state_weights, unimodal_states, unimodal_covariances):
        K, N, sd = state_weights.shape
        assert K == np.sum(self._enabled_models) and sd == self.state_dim
        if unimodal_states.is_cuda and not (torch.is_grad_enabled() and (
                state_weights.requires_grad or unimodal_states.requires_grad or unimodal_covariances.requires_grad)):
            return ops.kf_fuse_crossmodal(unimodal_states, unimodal_covariances, state_weights)
        mean = weighted_average(unimodal_states, state_weights)
        cw = state_weights[..., None] * state_weights[..., None, :]
        return mean, torch.sum(cw * unimodal_covariances, dim=0)

    def _state_weights(self, observations, N, device):
        on = self._enabled_models
        if np.sum(on) < len(on):
            w = _mask_weights(on, N, self.state_dim, device)
        else:
            w = self.crossmodal_weight_model(observations=observations)
        return w[on]

    def forward(self, *, observations, controls):
        N = controls.shape[0]
        K = int(np.sum(self._enabled_models))
        states, covs = self.calculate_unimodal_states(observations, controls)
        assert states.shape == (K, N, self.state_dim)
        assert covs.shape == (K, N, self.state_dim, self.state_dim)
        weights = self._state_weights(observations, N, states.device)
        assert weights.shape == (K, N, self.state_dim)
        mean, cov = self.calculate_weighted_states(weights, states, covs)
        assert mean.shape == (N, self.state_dim) and cov.shape == (N, self.state_dim, self.state_dim)
        self.weighted_covariances = cov
        for f in self.filter_models:  # quirk Q6: nobody reads these => no posterior feedback
            f.states_prev = mean
            f.states_covariance_prev = cov
        return mean

    def _sequence_weights(self, observations, T, N, device, grad=False):
        """(T, K_enabled, N, sd) fusion weights for a whole sequence; ``grad``: with autograd."""
        on = self._enabled_models
        if np.sum(on) < len(on):
            w = _mask_weights(on, N, self.state_dim, device)[on]
            return w[None].expand(T, *w.shape)
        wm = self.crossmodal_weight_model
        with torch.set_grad_enabled(grad):
            if hasattr(wm, "forward_sequence"):
                return wm.forward_sequence(observations, T, N)
            obs = SliceWrapper(observations)
            return torch.stack([wm(observations=obs[t]) for t in range(T)])

    def forward_loop(self, *, observations, controls):
        filters = self._enabled_filters()
        if isinstance(observations, dict) and self._train_fused(filters, controls, observations):
            # the F filters in one FusedEKFLoop; the (tiny) fusion stays torch expressions under autograd
            T, N = controls.shape[:2]
            assert SliceWrapper(observations).shape[:2] == (T, N)
            means, covs = self._advance_train(filters, controls, *self._sense_sequence_train(filters, observations, T, N))
            beta = self._sequence_weights(observations, T, N, controls.device, grad=True)
            beta = self._blackout_adjust(beta, observations).transpose(0, 1)  # (F,T,N,sd)
            cw = beta[..., None] * beta[..., None, :]
            self.weighted_covariances = torch.sum(cw * covs, dim=0)[-1]
            return weighted_average(means, beta)
        if not self._fusable(filters, controls) or tf_filters._has_hooks(self) or not isinstance(observations, dict):
            return super().forward_loop(observations=observations, controls=controls)
        T, N = controls.shape[:2]
        assert SliceWrapper(observations).shape[:2] == (T, N)
        zr = [f.sense_sequence(observations, T, N) for f in filters]
        z = torch.stack([a[0] for a in zr])
        r = torch.stack([a[1] for a in zr])
        means, covs = self._advance(filters, controls, z, r)          # (F,T,N,sd), (F,T,N,sd,sd)
        beta = self._sequence_weights(observations, T, N, controls.device)  # (T,F,N,sd)
        beta = self._blackout_adjust(beta, observations)
        fused_mean, fused_cov = ops.kf_fuse_crossmodal(means, covs, beta.transpose(0, 1).contiguous())
        self.weighted_covariances = fused_cov[-1]
        return fused_mean

    def _blackout_adjust(self, beta, observations):
        return beta

    def measurement_initialize_beliefs(self, observations):
        outs = [f.virtual_sensor_model(observations=observations) for f in self._enabled_filters()]
        weights = self.crossmodal_weight_model(observations=observations)[self._enabled_models]
        mean, cov = _measurement_level(torch.stack([o[0] for o in outs]), torch.stack([o[1] for o in outs]), weights)
        self.initialize_beliefs(mean=mean, covariance=cov)


def _information_fusion(states, covs):  # ref: base_models/unimodal_kf.py:199-242 (+1e-9 is elementwise)
    precision = torch.inverse(covs + 1e-9)
    cov = torch.inverse(precision.sum(dim=0) + 1e-9)
    return (cov @ (precision @ states[..., None]).sum(dim=0)).squeeze(-1)


class UnimodalKalmanFilter(_MultiFilter):
    """ref: crossmodal/base_models/unimodal_kf.py:118-270."""

    def forward(self, *, observations, controls):
        N = controls.shape[0]
        states, covs = self.calculate_unimodal_states(observations, controls)
        if states.shape[0] == 1:
            return states[0]
        if states.is_cuda and not (torch.is_grad_enabled() and (states.requires_grad or covs.requires_grad)):
            mean, _ = ops.kf_fuse_unimodal(states, covs)
        else:
            mean = _information_fusion(states, covs)
        assert mean.shape == (N, self.state_dim)
        return mean

    def forward_loop(self, *, observations, controls):
        filters = self._enabled_filters()
        if isinstance(observations, dict) and self._train_fused(filters, controls, observations):
            T, N = controls.shape[:2]
            assert SliceWrapper(observations).shape[:2] == (T, N)
            means, covs = self._advance_train(filters, controls, *self._sense_sequence_train(filters, observations, T, N))
            return means[0] if means.shape[0] == 1 else _information_fusion(means, covs)
        if not self._fusable(filters, controls) or tf_filters._has_hooks(self) or not isinstance(observations, dict):
            return super().forward_loop(observations=observations, controls=controls)
        T, N = controls.shape[:2]
        zr = [f.sense_sequence(observations, T, N) for f in filters]
        means, covs = self._advance(filters, controls, torch.stack([a[0] for a in zr]), torch.stack([a[1] for a in zr]))
        if means.shape[0] == 1:
            return means[0]
        return ops.kf_fuse_unimodal(means, covs)[0]


class CrossmodalVirtualSensorModel(tf_base.VirtualSensorModel, _EnabledModels):
    """R12, ref: crossmodal/base_models/crossmodal_kf.py:243-359."""

    def __init__(self, *, virtual_sensor_model, crossmodal_weight_model, state_dim: int):
        super().__init__(state_dim=state_dim)
        self.virtual_sensor_model = nn.ModuleList(virtual_sensor_model)
        self.crossmodal_weight_model = crossmodal_weight_model
        self._enabled_models = [True] * len(self.virtual_sensor_model)

    def forward(self, *, observations):
        on = self._enabled_models
        N = observations[[*observations][0]].shape[0]
        outs = [m(observations=observations) for m, flag in zip(self.virtual_sensor_model, on) if flag]
        states, trils = torch.stack([o[0] for o in outs]), torch.stack([o[1] for o in outs])
        if np.sum(on) < len(on):
            weights = _mask_weights(on, N, self.state_dim, states.device)
        else:
            weights = self.crossmodal_weight_model(observations=observations)
        if _fuse_kernel_ok(states, trils, weights):  # one launch: weighted mean, scaled covariance sum, Cholesky factor
            return ops.kf_fuse_measurements(states, trils, weights[on])
        mean, cov = _measurement_level(states, trils, weights[on])
        return mean, torch.linalg.cholesky(cov)


class UnimodalVirtualSensorModel(tf_base.VirtualSensorModel, _EnabledModels):
    """R12, ref: crossmodal/base_models/unimodal_kf.py:13-115 (returns a covariance, as the reference does)."""

    def __init__(self, *, virtual_sensor_model, state_dim: int):
        super().__init__(state_dim=state_dim)
        self.virtual_sensor_model = nn.ModuleList(virtual_sensor_model)
        self._enabled_models = [True] * len(self.virtual_sensor_model)

    def forward(self, *, observations):
        outs = [m(observations=observations) for m, flag in zip(self.virtual_sensor_model, self._enabled_models) if flag]
        states, trils = torch.stack([o[0] for o in outs]), torch.stack([o[1] for o in outs])
        if _fuse_kernel_ok(states, trils):
            return ops.kf_fuse_measurements(states, trils, None)
        covs = trils @ trils.transpose(-1, -2)
        if len(outs) == 1:
            return states[0], covs[0]
        precision = 1.0 / (trils + 1e-9)
        weights = torch.diagonal(precision, dim1=-2, dim2=-1)
        return weighted_average(states, weights), torch.inverse(precision.sum(dim=0) + 1e-9)


class _TaskCrossmodalKF(CrossmodalKalmanFilter):
    """Blackout-aware override, ref: crossmodal/door_models/crossmodal_kf.py:43-98 (quirk Q7)."""

    @staticmethod
    def _blackout_weights(raw, black):
        keep = (~black).float()[:, None]
        image = black.float()[:, None] * 1e-9 + keep * raw[0]
        force = black.float()[:, None] * (1.0 - 1e-9) + keep * raw[1]
        return torch.stack([image, force])

    def forward(self, *, observations, controls):
        if not self.know_image_blackout:
            return super().forward(observations=observations, controls=controls)
        black = _blackout_rows(observations)
        if torch.sum(black) == 0 or np.sum(self._enabled_models) < len(self._enabled_models):
            return super().forward(observations=observations, controls=controls)
        states, covs = self.calculate_unimodal_states(observations, controls)
        weights = self._blackout_weights(self.crossmodal_weight_model(observations=observations), black)
        mean, cov = self.calculate_weighted_states(weights, states, covs)
        self.weighted_covariances = cov
        return mean

    def _blackout_adjust(self, beta, observations):
        if not self.know_image_blackout or np.sum(self._enabled_models) < len(self._enabled_models):
            return beta
        img = observations["image"]
        black = img.reshape(*img.shape[:2], -1).abs().sum(dim=-1) < 1e-8  # (T, N)
        keep = (~black).float()[..., None]
        image = black.float()[..., None] * 1e-9 + keep * beta[:, 0]
        force = black.float()[..., None] * (1.0 - 1e-9) + keep * beta[:, 1]
        return torch.stack([image, force], dim=1)


def _make_kf_family(prefix, dyn_cls, sensor_cls, kf_cls, weight_cls, sd):
    def two_filters():
        return [kf_cls(dynamics_model=dyn_cls(), virtual_sensor_model=sensor_cls(modalities={"image"})),
                kf_cls(dynamics_model=dyn_cls(), virtual_sensor_model=sensor_cls(modalities={"pos", "sensors"}))]

    def two_sensors():
        return [sensor_cls(modalities={"image"}), sensor_cls(modalities={"pos", "sensors"})]

    def cross_init(self, know_image_blackout=False):
        CrossmodalKalmanFilter.__init__(self, filter_models=two_filters(),
                                        crossmodal_weight_model=weight_cls(state_dim=sd), state_dim=sd)
        self.know_image_blackout = know_image_blackout

    def uni_init(self):
        UnimodalKalmanFilter.__init__(self, filter_models=two_filters(), state_dim=sd)

    def mcross_init(self):
        kf_cls.__init__(self, dynamics_model=dyn_cls(), virtual_sensor_model=CrossmodalVirtualSensorModel(
            virtual_sensor_model=two_sensors(), crossmodal_weight_model=weight_cls(state_dim=sd), state_dim=sd))

    def muni_init(self):
        kf_cls.__init__(self, dynamics_model=dyn_cls(), virtual_sensor_model=UnimodalVirtualSensorModel(
            virtual_sensor_model=two_sensors(), state_dim=sd))

    return (
        type(prefix + "CrossmodalKalmanFilter", (_TaskCrossmodalKF,), {"__init__": cross_init}),
        type(prefix + "UnimodalKalmanFilter", (UnimodalKalmanFilter,), {"__init__": uni_init}),
        type(prefix + "MeasurementCrossmodalKalmanFilter", (kf_cls,), {"__init__": mcross_init}),
        type(prefix + "MeasurementUnimodalKalmanFilter", (kf_cls,), {"__init__": muni_init}),
    )


(PushCrossmodalKalmanFilter, PushUnimodalKalmanFilter, PushMeasurementCrossmodalKalmanFilter,
 PushMeasurementUnimodalKalmanFilter) = _make_kf_family(
    "Push", PushDynamicsModel, PushVirtualSensorModel, PushKalmanFilter, PushCrossmodalKalmanFilterWeightModel, 2)
(DoorCrossmodalKalmanFilter, DoorUnimodalKalmanFilter, DoorMeasurementCrossmodalKalmanFilter,
 DoorMeasurementUnimodalKalmanFilter) = _make_kf_family(
    "Door", DoorDynamicsModel, DoorVirtualSensorModel, DoorKalmanFilter, DoorCrossmodalKalmanFilterWeightModel, 3)

MODEL_TYPES = {
    "push": {c.__name__: c for c in (
        PushParticleFilter, PushCrossmodalParticleFilter, PushCrossmodalParticleFilterSeq5, PushUnimodalParticleFilter,
        PushKalmanFilter, PushCrossmodalKalmanFilter, PushUnimodalKalmanFilter,
        PushMeasurementCrossmodalKalmanFilter, PushMeasurementUnimodalKalmanFilter)},
    "door": {c.__name__: c for c in (
        DoorParticleFilter, DoorCrossmodalParticleFilter, DoorCrossmodalParticleFilterSeq5, DoorUnimodalParticleFilter,
        DoorKalmanFilter, DoorCrossmodalKalmanFilter, DoorUnimodalKalmanFilter,
        DoorMeasurementCrossmodalKalmanFilter, DoorMeasurementUnimodalKalmanFilter)},
}
