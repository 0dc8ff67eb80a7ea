"""``ParticleFilter`` / ``ExtendedKalmanFilter`` / ``VirtualSensorExtendedKalmanFilter`` with
torchfilter's public surface (SURVEY.md Appendix A.3, A.5; reference call sites
ref: crossmodal/push_models/pf.py:14-27, crossmodal/door_models/kf.py:14-28,
crossmodal/eval_helpers.py:125-142), executing in the sm_100a kernels of ``libmmf_b200.so``.

Dispatch (SURVEY.md section 8b):
  * recognised architectures (the reference's gated-residual dynamics and per-particle heads,
    see ``fused.py``) and no autograd  -> fully fused kernels, observation encoders hoisted over T;
  * training with frozen recognised dynamics -> the particle filter's ``training.FusedHeads`` / ``Reweight``, the
    Kalman filters' ``training.FusedEKFLoop`` (the recursion and its backward as one kernel each);
  * anything else (user-defined modules, or gradients required) -> the modules run as torch
    modules on the GPU and only the reweight / normalise / estimate / resample stages run in the
    kernels (torch ops where a gradient has to flow).
Extensions beyond upstream (all optional, defaults reproduce upstream behaviour):
  ``noise``          object supplying the random draws (``init_eps``, ``process_eps``,
                     ``resample_uniforms``) so that two implementations can be fed identical draws;
  ``resample_mode``  "multinomial" (upstream's inverse-CDF, torch.multinomial's CPU arithmetic),
                     "multinomial_fast", "systematic", "systematic_fast";
  ``precision``      "fp32" | "bf16x3" | "bf16" arithmetic of the per-particle MLP chain.
"""
import math
import warnings

import torch

from .. import _lib, fused, ops, training
from ..fannypack.utils import SliceWrapper
from .base import (
    DynamicsModel,
    Filter,
    KalmanFilterBase,
    KalmanFilterMeasurementModel,
    ParticleFilterMeasurementModel,
    VirtualSensorModel,
    require_cuda,
)

TIME_BATCHABLE = {
    # per-trajectory modules whose rows are independent, so (T, N, ...) can be run as one (T*N) batch
    "PushCrossmodalWeightModel", "DoorCrossmodalWeightModel", "PushVirtualSensorModel", "DoorVirtualSensorModel",
}


def _needs_grad(module, *tensors) -> bool:
    if not torch.is_grad_enabled():
        return False
    if any(t is not None and t.requires_grad for t in tensors):
        return True
    return any(p.requires_grad for p in module.parameters())


def _has_hooks(module) -> bool:
    """Forward hooks on the filter or on any sub-module (dynamics, measurement heads, encoders...): the fused loop
    never calls those modules' ``__call__``, so it must not be taken when somebody is listening."""
    return any(m._forward_hooks or m._forward_pre_hooks for m in module.modules())


class ParticleFilter(Filter):
    def __init__(
        self,
        *,
        dynamics_model: DynamicsModel,
        measurement_model: ParticleFilterMeasurementModel,
        num_particles: int = 100,
        resample=None,
        soft_resample_alpha: float = 1.0,
        estimation_method: str = "weighted_average",
    ):
        super().__init__(state_dim=dynamics_model.state_dim)
        assert isinstance(dynamics_model, DynamicsModel)
        assert isinstance(measurement_model, ParticleFilterMeasurementModel)
        self.dynamics_model = dynamics_model
        self.measurement_model = measurement_model
        self.num_particles = num_particles
        self.resample = resample
        self.soft_resample_alpha = soft_resample_alpha
        self.estimation_method = estimation_method
        self.particle_states = None
        self.particle_log_weights = None
        self._initialized = False
        # extensions
        self.noise = None
        self.resample_mode = "multinomial"
        self.precision = "bf16x3"
        self.debug = None  # set to a dict to capture intermediates of the last fused step
        # forward_loop on small problems is launch-bound (~15 launches + Python per step): the second call with the
        # same shapes captures the whole T-step recursion in a CUDA graph and later calls replay it
        self.graph_max_particles = 1 << 16  # N * M up to which forward_loop is graph-captured; 0 disables
        self.whole_loop = True  # forward_loop through mmf_pf_forward_loop (one C call); False: one kernel sequence per step
        self.fused_reweight = True  # training step: fusion / normalise / estimate and their backward as two kernels

    # ---- plan management -------------------------------------------------------------------------
    def fused_plan(self):
        # the cache holds the sub-modules themselves (compared by identity): a replaced module can never alias a
        # stale plan through a recycled id()
        cached = self.__dict__.get("_mmf_plan")
        if cached is None or cached[0] is not self.dynamics_model or cached[1] is not self.measurement_model:
            cached = (self.dynamics_model, self.measurement_model, fused.PFPlan.build(self))
            self.__dict__["_mmf_plan"] = cached
        return cached[2]

    # ---- random draws ------------------------------------------------------------------------------
    def _init_eps(self, M, N, sd, like):
        if self.noise is not None:
            return self.noise.init_eps(M, N, sd, like).to(like.device, torch.float32)
        return torch.randn((M, N, sd), device=like.device, dtype=torch.float32)

    def _process_eps(self, rows, sd, like):
        if self.noise is not None:
            return self.noise.process_eps(rows, sd, like).to(like.device, torch.float32)
        return torch.randn((rows, sd), device=like.device, dtype=torch.float32)

    def _uniforms(self, N, S, like, mode):
        if self.noise is not None:
            u = self.noise.resample_uniforms(N, S, like)
            return u.to(like.device, torch.float64)
        if ops.is_systematic(mode):
            return torch.rand((N,), device=like.device, dtype=torch.float64)
        return torch.rand((N * S,), device=like.device, dtype=torch.float64).reshape(N, S)

    # ---- A.3 initialize_beliefs (R2) ------------------------------------------------------------------
    def initialize_beliefs(self, *, mean: torch.Tensor, covariance: torch.Tensor) -> None:
        N = mean.shape[0]
        sd, M = self.state_dim, self.num_particles
        assert mean.shape == (N, sd)
        assert covariance.shape == (N, sd, sd)
        require_cuda(mean, "initialize_beliefs(mean=...)")
        eps = self._init_eps(M, N, sd, mean)
        self.particle_states, self.particle_log_weights = ops.pf_init(
            mean.detach().float(), covariance.detach().float().contiguous(), eps
        )
        self._initialized = True

    # ---- one step ----------------------------------------------------------------------------------------
    def _modes(self):
        resample = self.resample if self.resample is not None else (not self.training)
        mode = ops.RESAMPLE_MODES[self.resample_mode] if resample else ops.RESAMPLE_NONE
        assert self.estimation_method in ops.ESTIMATION, f"unknown estimation method {self.estimation_method}"
        return resample, mode

    def _retile_without_resampling(self):
        """A.3: particle count changed while resampling is off -> tile, pad with a random subset."""
        N, M, sd = self.particle_states.shape
        reps, extra = divmod(self.num_particles, M)
        idx = torch.arange(M, device=self.particle_states.device).repeat(reps)
        if extra:
            perm = self.noise.randperm(M) if self.noise is not None else torch.randperm(M)
            idx = torch.cat([idx, perm[:extra].to(idx.device)])
        self.particle_states = self.particle_states[:, idx, :].contiguous()
        logw = self.particle_log_weights[:, idx]
        self.particle_log_weights = (logw - torch.logsumexp(logw, dim=1, keepdim=True)).contiguous()

    def forward(self, *, observations, controls, _hoisted=None) -> torch.Tensor:
        assert self._initialized, "Particle filter not initialized: call initialize_beliefs() first"
        require_cuda(self.particle_states, "the particle set")
        resample, mode = self._modes()
        if not resample and self.num_particles != self.particle_states.shape[1]:
            self._retile_without_resampling()
        plan = self.fused_plan()
        grad = _needs_grad(self, self.particle_states, self.particle_log_weights)
        if plan is not None and not grad and isinstance(controls, torch.Tensor):
            return self._step_fused(plan, observations, controls, mode, _hoisted)
        if grad and isinstance(controls, torch.Tensor) and training.fused_train_applicable(self, plan, resample):
            return self._step_fused_train(plan, observations, controls, _hoisted)
        return self._step_generic(observations, controls, resample, mode, grad)

    def _head_rows(self, plan, observations, feats, rows_n):
        """(K, rows_n, 64): the observation half of every enabled head's first shared Linear (autograd on)."""
        rows = []
        for spec, on in zip(plan.heads, plan.enabled()):
            if not on:
                rows.append(self.particle_states.new_zeros((rows_n, fused.U)))
                continue
            mid = spec.shared[0]
            f = spec.observation_features(observations) if feats is None else feats[len(rows)]
            rows.append(torch.nn.functional.linear(f, mid.weight[:, : spec.feat_dim], mid.bias))
        return torch.stack(rows)

    def _step_fused_train(self, plan, observations, controls, hoisted=None, pre=None):
        """BPTT step (train mode: no resampling; dynamics frozen): kernels for the per-particle work and for fusion /
        normalisation / estimate, torch modules with autograd for the per-trajectory pieces.  ``pre`` = (dynamics row,
        head rows (K, N, 64), modality log-weights) when ``forward_loop`` computed them for the whole sequence."""
        states, logw = self.particle_states, self.particle_log_weights
        N, M, sd = states.shape
        enabled = plan.enabled()
        plan.refresh(states.device, backward=True)
        params = [p for spec in plan.heads for p in training.head_parameters(spec)]
        if pre is None:
            with torch.no_grad():
                dyn_row = ops.pf_traj_rows(plan.struct, plan.K, controls, [None] * plan.K)[0]
            head_rows = self._head_rows(plan, observations, None if hoisted is None else hoisted[0], N)
            modw = plan.modality_log_weights(observations) if hoisted is None else hoisted[1]
        else:
            dyn_row, head_rows, modw = pre
        eps = self._process_eps(N * M, sd, states)
        # one gradient token per autograd graph: the head parameters' gradients of all steps of a sequence are summed as
        # one flat tensor and distributed to the parameters once (training.HeadGradToken).  A carried log-weight without
        # grad_fn marks the start of a new graph (initialize_beliefs, or a detach for truncated BPTT): new token.
        tok = self.__dict__.get("_train_token")
        if tok is None or tok[0] is not plan or logw.grad_fn is None or not torch.is_grad_enabled():
            info = {"used": 0}
            tok = (plan, training.HeadGradToken.apply(plan, info, *params), info)
            self.__dict__["_train_token"] = tok
        moved, ll = training.FusedHeads.apply(plan, states, eps, dyn_row, head_rows, plan.enabled_mask(),
                                             ops.PRECISIONS[self.precision], tok[1], tok[2])
        if self.estimation_method == "weighted_average" and self.fused_reweight:
            # fusion over the enabled heads + reweight + normalise + estimate: one kernel, and one more for its backward
            logw_n, estimate = training.Reweight.apply(ll, modw, logw, moved, plan.enabled_mask())
            self.particle_states, self.particle_log_weights = moved, logw_n
            return estimate
        # select the enabled heads by slicing: indexing with a Python list would build the index tensor on the host and
        # copy it over (a synchronising H2D copy per step, and not capturable in a CUDA graph)
        on_idx = [k for k, on in enumerate(enabled) if on]
        all_on = len(on_idx) == len(enabled)
        ll = (ll if all_on else torch.stack([ll[k] for k in on_idx])).permute(1, 2, 0)  # (N, M, K_enabled)
        if modw is not None:
            mw = modw if all_on else torch.stack([modw[:, k] for k in on_idx], dim=1)
            ll = ll + mw[:, None, :]
        logw_unnorm = logw + torch.logsumexp(ll, dim=2)
        logw_n = logw_unnorm - torch.logsumexp(logw_unnorm, dim=1, keepdim=True)
        if self.estimation_method == "weighted_average":
            estimate = torch.sum(torch.exp(logw_n)[:, :, None] * moved, dim=1)
        else:
            best = torch.argmax(logw_n, dim=1)
            estimate = moved[torch.arange(N, device=best.device), best]
        self.particle_states, self.particle_log_weights = moved, logw_n
        return estimate

    def _step_fused(self, plan, observations, controls, mode, hoisted):
        states, logw = self.particle_states, self.particle_log_weights
        N, M, sd = states.shape
        with torch.no_grad():
            if hoisted is None:
                feats = plan.head_features(observations)
                modw = plan.modality_log_weights(observations)
            else:
                feats, modw = hoisted
            eps = self._process_eps(N * M, sd, states)
            uniforms = self._uniforms(N, self.num_particles, states, mode) if mode != ops.RESAMPLE_NONE else None
            out = plan.step(
                states, logw, controls, feats, modw, eps,
                precision=ops.PRECISIONS[self.precision], estimation=ops.ESTIMATION[self.estimation_method],
                mode=mode, alpha=self.soft_resample_alpha, M_out=self.num_particles, uniforms=uniforms,
                want_debug=self.debug is not None,
            )
        self.particle_states, self.particle_log_weights = out["states"], out["logw"]
        if self.debug is not None:
            self.debug.clear()
            self.debug.update(out, eps=eps, uniforms=uniforms)
        return out["estimate"]

    def _step_generic(self, observations, controls, resample, mode, grad):
        states, logw = self.particle_states, self.particle_log_weights
        N, M, sd = states.shape
        flat_controls = SliceWrapper(controls).map(lambda c: c.repeat_interleave(M, dim=0))
        pred, trils = self.dynamics_model(initial_states=states.reshape(-1, sd), controls=flat_controls)
        eps = self._process_eps(N * M, sd, states)
        moved = (pred + (trils @ eps[..., None]).squeeze(-1)).view(N, M, sd)
        logw_unnorm = logw + self.measurement_model(states=moved, observations=observations)
        assert logw_unnorm.shape == (N, M)
        uniforms = self._uniforms(N, self.num_particles, states, mode) if resample else None
        if not grad:
            out = ops.pf_normalize_resample(
                moved.detach(), logw_unnorm.detach(), estimation=ops.ESTIMATION[self.estimation_method], mode=mode,
                alpha=self.soft_resample_alpha, M_out=self.num_particles, uniforms=uniforms,
            )
            self.particle_states, self.particle_log_weights = out["states"], out["logw"]
            return out["estimate"]
        # gradient path: differentiable torch ops; only the (non-differentiable) index draw is a kernel
        logw_n = logw_unnorm - torch.logsumexp(logw_unnorm, dim=1, keepdim=True)
        if self.estimation_method == "weighted_average":
            estimate = torch.sum(torch.exp(logw_n)[:, :, None] * moved, dim=1)
        else:
            best = torch.argmax(logw_n, dim=1)
            estimate = moved[torch.arange(N, device=best.device), best]
        if resample:
            alpha = self.soft_resample_alpha
            uniform_lw = logw_n.new_full((N, self.num_particles), -math.log(M))
            if alpha < 1.0:
                assert self.num_particles == M
                logits = torch.logsumexp(
                    torch.stack([logw_n + math.log(alpha), uniform_lw + math.log(1.0 - alpha)]), dim=0
                )
                new_logw = logw_n - logits
            else:
                logits, new_logw = logw_n, uniform_lw
            idx = ops.resample_indices(logits.detach().contiguous(), uniforms, mode=mode, M_out=self.num_particles)
            moved = torch.gather(moved, 1, idx[:, :, None].expand(N, self.num_particles, sd))
            logw_n = torch.gather(new_logw, 1, idx) if alpha < 1.0 else new_logw
        self.particle_states, self.particle_log_weights = moved, logw_n
        return estimate

    # ---- whole sequence (R1) -----------------------------------------------------------------------------
    def forward_loop(self, *, observations, controls) -> torch.Tensor:
        plan = self.fused_plan()
        if (
            plan is None
            or not self._initialized
            or not isinstance(controls, torch.Tensor)
            or not isinstance(observations, dict)
            or _has_hooks(self)
        ):
            return super().forward_loop(observations=observations, controls=controls)
        if _needs_grad(self, self.particle_states, self.particle_log_weights):
            resample, _ = self._modes()
            T, N = controls.shape[:2]
            if (T == 0 or not controls.is_cuda or not training.fused_train_applicable(self, plan, resample)
                    or self.num_particles != self.particle_states.shape[1]
                    or not all(isinstance(v, torch.Tensor) and v.is_cuda for v in observations.values())):
                return super().forward_loop(observations=observations, controls=controls)
            # training: encoders, weight model and the heads' observation rows once over all T * N rows, with autograd
            flat = fused.flatten_time(observations, T, N)
            feats = [spec.observation_features(flat) if on else None for spec, on in zip(plan.heads, plan.enabled())]
            wm = getattr(plan.mm, "crossmodal_weight_model", None) if plan.composite else None
            if wm is None:
                modw = None
            elif type(wm).__name__ in TIME_BATCHABLE or getattr(wm, "_mmf_time_batchable", False):
                modw = plan.modality_log_weights(flat)
            else:  # a user weight model may couple the rows of a batch: one call per step, as the reference does
                obs = SliceWrapper(observations)
                modw = torch.stack([plan.modality_log_weights(obs[t]) for t in range(T)])
            return self.forward_loop_train_hoisted(feats, modw, controls)
        require_cuda(controls, "controls")
        T, N = controls.shape[:2]
        assert SliceWrapper(observations).shape[:2] == (T, N), "observations and controls disagree on (T, N)"
        if all(isinstance(v, torch.Tensor) and v.device.type == "cpu" for v in observations.values()):
            # host (pinned) observations: stream them in behind the encoders instead of copying first
            observations = fused.StagedObservations(observations, controls.device, T, N, chunk_rows=16384)
        feats, modw = self.hoist_observations(plan, observations, T, N)
        if isinstance(observations, fused.StagedObservations):
            observations.ready(T * N)
        return self.forward_loop_hoisted(feats, modw, controls)

    def forward_loop_train_hoisted(self, feats, modw, controls) -> torch.Tensor:
        """BPTT over a sequence with everything that does not depend on the particles computed ONCE for all T steps
        (SURVEY.md section 8f rank 1, training side): the observation halves of the heads' first shared Linear
        (``feats``: K tensors (T, N, F_k) of observation features, gradients welcome), the dynamics rows of all steps
        (one ``mmf_pf_traj_rows`` launch) and the modality log-weights ``modw`` (T, N, K) | None.  Per step only the
        per-particle kernels (``FusedHeads``) and the reweight kernels (``Reweight``) remain.  Same numbers as T calls of
        ``forward``."""
        plan = self.fused_plan()
        T, N = controls.shape[:2]
        plan.refresh(controls.device, backward=True)
        flat = [None if f is None else f.reshape(T * N, -1) for f in feats]
        rows_all = self._head_rows(plan, None, flat, T * N).view(plan.K, T, N, fused.U).unbind(1)
        with torch.no_grad():
            dyn_rows = ops.pf_traj_rows(plan.struct, plan.K, controls.reshape(T * N, -1), [None] * plan.K)[0].view(T, N, fused.U)
        modw_t = [None] * T if modw is None else modw.reshape(T, N, -1).unbind(0)
        estimates = []
        for t in range(T):
            estimates.append(self._step_fused_train(plan, None, controls[t], pre=(dyn_rows[t], rows_all[t], modw_t[t])))
        return torch.stack(estimates)

    def forward_loop_hoisted(self, feats, modw, controls) -> torch.Tensor:
        """The recursion proper, given the per-head observation features (T, N, F_k) and modality log-weights
        (T, N, K) of ``hoist_observations``: CUDA-graph replay for small problems, otherwise ONE C call that enqueues the
        per-trajectory rows of all steps plus two kernels per step (``mmf_pf_forward_loop``); the per-step path remains
        for what that call does not cover (debug capture, soft resampling, a changing particle count)."""
        T, N = controls.shape[:2]
        replayed = self._forward_loop_graph(feats, modw, controls, T, N)
        if replayed is not None:
            return replayed
        whole = self._forward_loop_whole(feats, modw, controls, T, N)
        if whole is not None:
            return whole
        estimates = controls.new_zeros((T, N, self.state_dim), dtype=torch.float32)
        for t in range(T):
            hoisted = ([None if f is None else f[t] for f in feats], None if modw is None else modw[t])
            estimates[t] = self.forward(observations=None, controls=controls[t], _hoisted=hoisted)
        return estimates

    def _forward_loop_whole(self, feats, modw, controls, T, N):
        """``mmf_pf_forward_loop``: returns the estimates, or None when the per-step path has to run."""
        resample, mode = self._modes()
        M = self.particle_states.shape[1]
        if (
            not self.whole_loop or self.debug is not None or T == 0 or controls.dtype != torch.float32
            or self.num_particles != M or (resample and self.soft_resample_alpha < 1.0)
            or self.precision not in ops.PRECISIONS
        ):
            return None
        plan = self.fused_plan()
        sd = self.state_dim
        like = self.particle_states
        with torch.no_grad():
            plan.refresh(like.device)
            if self.noise is not None:  # injected draws: same per-step protocol as the step-by-step path
                eps = torch.stack([self._process_eps(N * M, sd, like) for _ in range(T)])
                uniforms = torch.stack([self._uniforms(N, M, like, mode) for _ in range(T)]) if resample else None
            else:
                eps = torch.randn((T, N * M, sd), device=like.device, dtype=torch.float32)
                uniforms = None
                if resample:
                    shape = (T, N) if ops.is_systematic(mode) else (T, N, M)
                    uniforms = torch.rand(shape, device=like.device, dtype=torch.float64)
            states = like.detach().clone()  # the reference rebinds particle_states every step: never mutate the caller's tensor
            logw = self.particle_log_weights.detach().clone()
            est = ops.pf_forward_loop(
                plan.struct, states, logw, controls, feats, modw, plan.enabled_mask(), eps,
                precision=ops.PRECISIONS[self.precision], estimation=ops.ESTIMATION[self.estimation_method], mode=mode,
                uniforms=uniforms,
            )
        self.particle_states, self.particle_log_weights = states, logw
        return est

    def _forward_loop_graph(self, feats, modw, controls, T, N):
        """CUDA-graph replay of the hoisted T-step recursion (SURVEY.md section 8f rank 2).  Returns the estimates,
        or None when the loop has to run eagerly (large problem, injected noise, debug capture, first sight of a
        configuration, or a capture that failed once)."""
        M_in = self.particle_states.shape[1]
        if (
            not self.graph_max_particles
            or N * max(M_in, self.num_particles) > self.graph_max_particles
            or self.noise is not None
            or self.debug is not None
            or controls.dtype != torch.float32
        ):
            return None
        resample, mode = self._modes()
        if not resample and self.num_particles != M_in:
            return None
        key = (
            T, N, M_in, self.num_particles, self.state_dim, str(controls.device), tuple(controls.shape), mode,
            self.estimation_method, float(self.soft_resample_alpha), self.precision,
            tuple(None if f is None else tuple(f.shape) for f in feats), None if modw is None else tuple(modw.shape),
            tuple(self.fused_plan().enabled()), tuple((p.data_ptr(), p._version) for p in self.parameters()),
        )
        cache = self.__dict__.setdefault("_mmf_loop_graph", {"key": None, "graph": None, "static": None})
        if cache["key"] != key:
            cache.update(key=key, graph=None, static=None)  # first sight: run eagerly (also warms every launcher)
            return None
        if cache["graph"] is False:
            return None
        if cache["graph"] is None:
            st = {
                "feats": [None if f is None else f.clone() for f in feats],
                "modw": None if modw is None else modw.clone(),
                "controls": controls.clone(),
                "states0": self.particle_states.detach().clone(),
                "logw0": self.particle_log_weights.detach().clone(),
                "est": controls.new_zeros((T, N, self.state_dim), dtype=torch.float32),
            }
            live = (self.particle_states, self.particle_log_weights)
            graph = torch.cuda.CUDAGraph()
            launches_before = ops.PROFILE.launches
            try:
                self.particle_states, self.particle_log_weights = st["states0"], st["logw0"]
                with torch.cuda.graph(graph):
                    whole = self._forward_loop_whole(st["feats"], st["modw"], st["controls"], T, N)
                    if whole is not None:  # 1 + 2 T kernels + the two noise draws
                        st["est"] = whole
                    else:
                        for t in range(T):
                            hoisted = ([None if f is None else f[t] for f in st["feats"]],
                                       None if st["modw"] is None else st["modw"][t])
                            st["est"][t] = self.forward(observations=None, controls=st["controls"][t], _hoisted=hoisted)
                st["statesT"], st["logwT"] = self.particle_states, self.particle_log_weights
                # kernels recorded into the graph: they run at every replay, not during capture
                st["launches"] = ops.PROFILE.launches - launches_before
                ops.PROFILE.launches = launches_before
            except Exception as exc:  # capture is an optimisation: never let it take the eager path down with it
                self.particle_states, self.particle_log_weights = live
                cache.update(graph=False, static=None)
                torch.cuda.synchronize()
                warnings.warn(f"forward_loop: CUDA-graph capture failed ({type(exc).__name__}: {exc}); "
                              "this configuration keeps running with eager launches", RuntimeWarning)
                return None
            self.particle_states, self.particle_log_weights = live
            cache.update(graph=graph, static=st)
        st = cache["static"]
        for dst, src in zip(st["feats"], feats):
            if dst is not None:
                dst.copy_(src)
        if st["modw"] is not None:
            st["modw"].copy_(modw)
        st["controls"].copy_(controls)
        st["states0"].copy_(self.particle_states)
        st["logw0"].copy_(self.particle_log_weights)
        cache["graph"].replay()
        ops.PROFILE.launches += st["launches"]
        self.particle_states = st["statesT"].clone()
        self.particle_log_weights = st["logwT"].clone()
        return st["est"].clone()

    def hoist_observations(self, plan, observations, T, N):
        """The observation encoders and the weight model do not depend on the particles: run them
        once over all T*N rows (SURVEY.md section 8f rank 1) instead of once per step per model."""
        with torch.no_grad():
            enabled = plan.enabled()
            feats = []
            for h, on in zip(plan.heads, enabled):
                if not on:
                    feats.append(None)
                    continue
                chunks = fused.batched_over_time(h.observation_features, observations, T, N)
                feats.append(torch.cat(chunks).reshape(T, N, -1).contiguous())
            wm = getattr(plan.mm, "crossmodal_weight_model", None) if plan.composite else None
            if wm is None:
                modw = None
            elif type(wm).__name__ in TIME_BATCHABLE or getattr(wm, "_mmf_time_batchable", False):
                chunks = fused.batched_over_time(lambda o: wm(observations=o), observations, T, N)
                modw = torch.cat(chunks).reshape(T, N, -1).contiguous()
            else:
                if isinstance(observations, fused.StagedObservations):
                    observations.ready(T * N)
                obs = SliceWrapper(observations)
                modw = torch.stack([wm(observations=obs[t]) for t in range(T)]).contiguous()
        return feats, modw


class ExtendedKalmanFilter(KalmanFilterBase):
    """A.5 for arbitrary user models (torch ops on the GPU).  The fused kernel path lives in
    ``VirtualSensorExtendedKalmanFilter``, the only EKF flavour the reference instantiates."""

    def _predict_step(self, *, controls):
        mean, cov = self._belief_mean, self._belief_covariance
        pred, q_tril = self.dynamics_model(initial_states=mean, controls=controls)
        A = self.dynamics_model.jacobian(initial_states=mean, controls=controls)
        self._belief_mean = pred
        self._belief_covariance = A @ cov @ A.transpose(-1, -2) + q_tril @ q_tril.transpose(-1, -2)

    def _update_step(self, *, observations):
        mean, cov = self._belief_mean, self._belief_covariance
        expected, r_tril = self.measurement_model(states=mean)
        Cm = self.measurement_model.jacobian(states=mean)
        S = Cm @ cov @ Cm.transpose(-1, -2) + r_tril @ r_tril.transpose(-1, -2)
        gain = cov @ Cm.transpose(-1, -2) @ torch.inverse(S)
        self._belief_mean = mean + (gain @ (observations - expected)[:, :, None]).squeeze(-1)
        eye = torch.eye(self.state_dim, device=cov.device, dtype=cov.dtype)
        self._belief_covariance = (eye - gain @ Cm) @ cov


class _IdentityMeasurementModel(KalmanFilterMeasurementModel):
    def __init__(self, *, state_dim: int):
        super().__init__(state_dim=state_dim, observation_dim=state_dim)
        self.scale_tril = None

    def forward(self, *, states):
        assert self.scale_tril is not None
        return states, self.scale_tril

    def jacobian(self, *, states):
        eye = torch.eye(self.state_dim, device=states.device, dtype=states.dtype)
        return eye[None].expand(states.shape[0], self.state_dim, self.state_dim)


class VirtualSensorExtendedKalmanFilter(ExtendedKalmanFilter):
    def __init__(self, *, dynamics_model: DynamicsModel, virtual_sensor_model: VirtualSensorModel):
        super().__init__(
            dynamics_model=dynamics_model,
            measurement_model=_IdentityMeasurementModel(state_dim=dynamics_model.state_dim),
        )
        self.virtual_sensor_model = virtual_sensor_model
        self.fused_train = True  # training with frozen dynamics: the recursion and its backward as one kernel each

    def fused_plan(self):
        cached = self.__dict__.get("_mmf_plan")
        if cached is None or cached[0] is not self.dynamics_model:
            cached = (self.dynamics_model, fused.EKFPlan.build([self]))
            self.__dict__["_mmf_plan"] = cached
        return cached[1]

    def _use_fused(self, controls):
        return (
            isinstance(controls, torch.Tensor)
            and self.fused_plan() is not None
            and not _needs_grad(self, self._belief_mean, self._belief_covariance)
        )

    def _train_fused(self, observations, controls):
        return self._initialized and training.fused_ekf_train_applicable(
            self, [self], self.fused_plan(), controls, observations, (self._belief_mean, self._belief_covariance))

    def _advance_train(self, controls, z, r_tril):
        """Training step(s) through ``training.FusedEKFLoop``: controls (T,N,cd), z (T,N,sd), r_tril (T,N,sd,sd) ->
        posterior means (T,N,sd).  The new belief keeps its ``grad_fn``, so the next call chains the gradient."""
        means, covs = training.FusedEKFLoop.apply(self.fused_plan(), self._belief_mean[None], self._belief_covariance[None],
                                                  controls, z[None], r_tril[None])
        self._belief_mean, self._belief_covariance = means[0, -1], covs[0, -1]
        return means[0]

    def forward(self, *, observations, controls):
        assert self._initialized, "Kalman filter not initialized: call initialize_beliefs() first"
        require_cuda(self._belief_mean, "the belief mean")
        z, r_tril = self.virtual_sensor_model(observations=observations)
        if self._train_fused(observations, controls):
            assert controls.shape[0] == self._belief_mean.shape[0]
            return self._advance_train(controls[None], z[None], r_tril[None])[0]
        if not self._use_fused(controls):
            self.measurement_model.scale_tril = r_tril
            return super().forward(observations=z, controls=controls)
        assert controls.shape[0] == self._belief_mean.shape[0]
        means, covs = self.fused_plan().loop(
            self._belief_mean.detach()[None], self._belief_covariance.detach()[None].contiguous(),
            controls[None], z.detach()[None, None], r_tril.detach()[None, None],
        )
        self._belief_mean, self._belief_covariance = means[0, 0], covs[0, 0]
        return self._belief_mean

    def sense_sequence(self, observations, T, N, grad=False):
        """Virtual-sensor outputs for all T steps: z (T,N,sd), r_tril (T,N,sd,sd); ``grad``: with autograd."""
        vs = self.virtual_sensor_model
        with torch.set_grad_enabled(grad):
            if type(vs).__name__ in TIME_BATCHABLE or getattr(vs, "_mmf_time_batchable", False):
                outs = fused.batched_over_time(lambda o: vs(observations=o), observations, T, N)
                z = torch.cat([o[0] for o in outs]).reshape(T, N, -1)
                r = torch.cat([o[1] for o in outs]).reshape(T, N, self.state_dim, self.state_dim)
            else:
                obs = SliceWrapper(observations)
                outs = [vs(observations=obs[t]) for t in range(T)]
                z = torch.stack([o[0] for o in outs])
                r = torch.stack([o[1] for o in outs])
        return z.contiguous(), r.contiguous()

    def forward_loop(self, *, observations, controls):
        if isinstance(observations, dict) and self._train_fused(observations, controls):
            T, N = controls.shape[:2]
            assert SliceWrapper(observations).shape[:2] == (T, N), "observations and controls disagree on (T, N)"
            z, r_tril = self.sense_sequence(observations, T, N, grad=True)
            return self._advance_train(controls, z, r_tril)
        if not self._initialized or not self._use_fused(controls) or _has_hooks(self) or not isinstance(observations, dict):
            return super().forward_loop(observations=observations, controls=controls)
        require_cuda(controls, "controls")
        T, N = controls.shape[:2]
        assert SliceWrapper(observations).shape[:2] == (T, N), "observations and controls disagree on (T, N)"
        z, r_tril = self.sense_sequence(observations, T, N)
        means, covs = self.fused_plan().loop(
            self._belief_mean.detach()[None], self._belief_covariance.detach()[None].contiguous(),
            controls, z[None], r_tril[None],
        )
        self._belief_mean, self._belief_covariance = means[0, -1], covs[0, -1]
        return means[0]
