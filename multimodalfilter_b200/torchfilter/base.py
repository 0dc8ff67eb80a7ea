"""Base classes with torchfilter's constructor / forward signatures (SURVEY.md Appendix A.1, A.2,
A.4), so the reference's model definitions subclass them unchanged
(ref: crossmodal/push_models/dynamics.py:10-14, crossmodal/base_models/crossmodal_pf.py:33-49,
crossmodal/door_models/kf.py:31-41).

These are interface + bookkeeping only; the recursion that runs on them lives in ``filters.py``
and executes in CUDA kernels.  Tensors must be on a CUDA device: there is no CPU path.
"""
import abc

import torch
import torch.nn as nn

from .. import _lib
from ..fannypack.utils import SliceWrapper


def require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise _lib.MMFError(
            f"{what} is on '{t.device}': multimodalfilter_b200 runs the filter recursion in sm_100a CUDA "
            "kernels and has no CPU fallback; move the model and its inputs to a B200"
        )


class Filter(nn.Module, abc.ABC):
    def __init__(self, *, state_dim: int):
        super().__init__()
        self.state_dim = state_dim

    @abc.abstractmethod
    def initialize_beliefs(self, *, mean: torch.Tensor, covariance: torch.Tensor) -> None:
        ...

    @abc.abstractmethod
    def forward(self, *, observations, controls) -> torch.Tensor:
        ...

    def forward_loop(self, *, observations, controls) -> torch.Tensor:
        """A.2: (T, N, ...) inputs -> (T, N, state_dim) estimates, one ``__call__`` per step so that
        forward hooks keep firing.  Filters with a whole-sequence fused path override this."""
        obs, ctrl = SliceWrapper(observations), SliceWrapper(controls)
        T, N = ctrl.shape[:2]
        assert obs.shape[:2] == (T, N), "observations and controls disagree on (T, N)"
        estimates = None
        for t in range(T):
            step = self(observations=obs[t], controls=ctrl[t])
            if estimates is None:
                assert step.shape == (N, self.state_dim)
                estimates = step.new_zeros((T, N, self.state_dim))
            estimates[t] = step
        return estimates


class DynamicsModel(nn.Module, abc.ABC):
    def __init__(self, *, state_dim: int):
        super().__init__()
        self.state_dim = state_dim

    @abc.abstractmethod
    def forward(self, *, initial_states, controls):
        """-> (predicted states (N, sd), scale_tril (N, sd, sd))"""

    def forward_loop(self, *, initial_states, controls):
        """Open-loop rollout (used at ref: crossmodal/eval_helpers.py:135-137).  Recognised gated-residual dynamics with
        CUDA fp32 inputs run the T steps in one kernel launch (and, when a gradient is needed, the reverse mode in one
        more: ``training.dynamics_rollout``); anything else runs the modules step by step."""
        ctrl = SliceWrapper(controls)
        T, N = ctrl.shape[:2]
        assert initial_states.shape == (N, self.state_dim)
        from .. import training

        states = training.dynamics_rollout(self, initial_states, controls)
        if states is not None:
            q = self.Q_scale_tril if hasattr(self, "Q_scale_tril") else torch.diag(self.Q_scale_tril_diag)
            return states, q.expand(T, N, self.state_dim, self.state_dim).contiguous()
        states, trils, x = [], [], initial_states
        for t in range(T):
            x, tril = self(initial_states=x, controls=ctrl[t])
            states.append(x)
            trils.append(tril)
        return torch.stack(states), torch.stack(trils)

    def jacobian(self, *, initial_states, controls) -> torch.Tensor:
        """A.4: (N, sd, sd) with A[n, i, j] = d f_i / d x_j.

        Recognised gated-residual dynamics evaluated without autograd use the forward-mode CUDA
        kernel (``mmf_dynamics_jacobian``); otherwise (training through the Jacobian, or a
        user-defined model) the reference's reverse-mode construction runs as torch ops."""
        if not torch.is_grad_enabled() and isinstance(controls, torch.Tensor) and initial_states.is_cuda:
            from .. import fused

            plan = self.__dict__.get("_mmf_jac_plan")
            if plan is None:
                plan = fused.EKFPlan.build([_DynamicsHolder(self)]) or False
                self.__dict__["_mmf_jac_plan"] = plan
            if plan:
                return plan.jacobian(0, initial_states, controls)[1]
        with torch.enable_grad():
            N, sd = initial_states.shape
            x = initial_states.detach()[:, None, :].repeat(1, sd, 1).requires_grad_(True)
            u = SliceWrapper(controls).map(lambda c: c.repeat_interleave(sd, dim=0))
            pred, _ = self(initial_states=x.reshape(N * sd, sd), controls=u)
            seed = torch.eye(sd, device=pred.device, dtype=pred.dtype).repeat(N, 1, 1)
            (jac,) = torch.autograd.grad(pred.reshape(N, sd, sd), x, seed, create_graph=True)
        return jac


class _DynamicsHolder:
    def __init__(self, dynamics_model):
        self.dynamics_model = dynamics_model


class ParticleFilterMeasurementModel(nn.Module, abc.ABC):
    def __init__(self, *, state_dim: int):
        super().__init__()
        self.state_dim = state_dim

    @abc.abstractmethod
    def forward(self, *, states, observations) -> torch.Tensor:
        """states (N, M, sd) -> log-likelihoods (N, M)"""


class KalmanFilterMeasurementModel(nn.Module, abc.ABC):
    def __init__(self, *, state_dim: int, observation_dim: int):
        super().__init__()
        self.state_dim = state_dim
        self.observation_dim = observation_dim

    @abc.abstractmethod
    def forward(self, *, states):
        """states (N, sd) -> (expected observations (N, od), scale_tril (N, od, od))"""

    def jacobian(self, *, states) -> torch.Tensor:
        with torch.enable_grad():
            N, sd = states.shape
            od = self.observation_dim
            x = states.detach()[:, None, :].repeat(1, od, 1).requires_grad_(True)
            pred, _ = self(states=x.reshape(N * od, sd))
            seed = torch.eye(od, device=pred.device, dtype=pred.dtype).repeat(N, 1, 1)
            (jac,) = torch.autograd.grad(pred.reshape(N, od, od), x, seed, create_graph=True)
        return jac


class VirtualSensorModel(nn.Module, abc.ABC):
    def __init__(self, *, state_dim: int):
        super().__init__()
        self.state_dim = state_dim

    @abc.abstractmethod
    def forward(self, *, observations):
        """-> (virtual observation z (N, sd), scale_tril (N, sd, sd))"""


class KalmanFilterBase(Filter, abc.ABC):
    """Gaussian belief (``_belief_mean``, ``_belief_covariance``; the latter is read directly at
    ref: crossmodal/base_models/crossmodal_kf.py:180)."""

    def __init__(self, *, dynamics_model: DynamicsModel, measurement_model: KalmanFilterMeasurementModel):
        super().__init__(state_dim=dynamics_model.state_dim)
        assert isinstance(dynamics_model, DynamicsModel)
        assert isinstance(measurement_model, KalmanFilterMeasurementModel)
        self.dynamics_model = dynamics_model
        self.measurement_model = measurement_model
        self._belief_mean = None
        self._belief_covariance = None
        self._initialized = False

    @property
    def belief_mean(self):
        return self._belief_mean

    @belief_mean.setter
    def belief_mean(self, value):
        assert value.dim() == 2 and value.shape[1] == self.state_dim
        self._belief_mean = value

    @property
    def belief_covariance(self):
        return self._belief_covariance

    @belief_covariance.setter
    def belief_covariance(self, value):
        assert value.dim() == 3 and value.shape[1:] == (self.state_dim, self.state_dim)
        self._belief_covariance = value

    def initialize_beliefs(self, *, mean, covariance):
        N = mean.shape[0]
        assert mean.shape == (N, self.state_dim)
        assert covariance.shape == (N, self.state_dim, self.state_dim)
        self.belief_mean = mean
        self.belief_covariance = covariance
        self._initialized = True

    def forward(self, *, observations, controls):
        assert self._initialized, "Kalman filter not initialized: call initialize_beliefs() first"
        assert SliceWrapper(controls).shape[0] == self._belief_mean.shape[0]
        self._predict_step(controls=controls)
        self._update_step(observations=observations)
        return self.belief_mean

    @abc.abstractmethod
    def _predict_step(self, *, controls):
        ...

    @abc.abstractmethod
    def _update_step(self, *, observations):
        ...
