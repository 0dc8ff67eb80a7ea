"""BPTT support: the fused training step of the particle filter (BASELINE config C4), and ``FusedEKFLoop``, the
extended Kalman filters' recursion and its reverse mode in one launch each.

In train mode torchfilter does not resample (A.3) and every curriculum of the reference freezes the
dynamics before end-to-end training (ref: scripts/push_task/train_push.py:154,213), so the particle
states carry no gradient to a trainable leaf; the loss reaches the parameters only through the
log-weights.  One training step is therefore

    moved, ll_k = kernel(states, eps, rows)            forward:  mmf_pf_heads_forward_train
    d ll_k -> delta of every head layer                backward: mmf_pf_heads_backward
    dW = delta^T a, db = sum delta, d rows_k = sum_m delta_mid      (reductions over the N*M rows)

wrapped in one ``torch.autograd.Function``; the fusion log-sum-exp, the normalisation and the
estimate are (N, M)-sized torch ops that autograd differentiates itself, and the per-trajectory
pieces (observation encoders, the observation half of the first shared Linear, the modality weight
model) stay ordinary torch modules, so their gradients come from autograd as well.
"""
from typing import List

import torch

from . import _lib, ops

U = _lib.UNITS


def head_parameters(spec) -> List[torch.Tensor]:
    """Trainable tensors of one head's per-particle chain, in a fixed order (see ``_grads_for_head``)."""
    (in_lin, pre), (mid, post, out) = spec.state, spec.shared
    ps = [in_lin.weight, in_lin.bias]
    for r in pre:
        ps += [r.block1.weight, r.block1.bias, r.block2.weight, r.block2.bias]
    ps += [mid.weight]
    for r in post:
        ps += [r.block1.weight, r.block1.bias, r.block2.weight, r.block2.bias]
    ps += [out.weight, out.bias]
    return ps


def mid_layer_index(spec) -> int:
    return 2 * len(spec.state[1])


def _grads_for_head(spec, dW, db, g_in, g_out, d_ll_sum):
    """dW (L, 64, 64), db (L+1, 64), g_in (64, sd), g_out (64,) from mmf_pf_heads_weight_grads; d_ll_sum (1,) = the sum
    of d ll over the particles (gradient of the output bias).  Returns grads in head_parameters order and the index of
    the mid layer."""
    (in_lin, pre), (mid, post, out) = spec.state, spec.shared
    L = 2 * len(pre) + 1 + 2 * len(post)
    grads = [g_in, db[L]]
    layer = 0
    for _ in pre:
        for _half in range(2):
            grads += [dW[layer], db[layer]]
            layer += 1
    g_mid = torch.zeros_like(mid.weight)
    g_mid[:, spec.feat_dim:] = dW[layer]  # state half; the observation half flows through the rows
    grads += [g_mid]
    mid_layer = layer
    layer += 1
    for _ in post:
        for _half in range(2):
            grads += [dW[layer], db[layer]]
            layer += 1
    grads += [g_out[None, :], d_ll_sum.reshape(1)]
    return grads, mid_layer


class HeadGradToken(torch.autograd.Function):
    """All head parameters of a plan -> ONE flat tensor whose only purpose is to carry gradients: ``FusedHeads`` takes the
    token instead of the ~30 parameters per head and hands its backward the per-step parameter gradients as one flat
    tensor [dW | db | g_in | g_out | sum d_ll] per head.  Over a T-step sequence autograd then sums T flat tensors (T - 1
    adds) and this node distributes the total to the parameters ONCE, instead of 61 ``AccumulateGrad`` additions per
    filter step (915 small kernels per C4 training step).  Heads that no step of the sequence enabled get ``None``."""

    @staticmethod
    def forward(ctx, plan, info, *params):
        ctx.plan, ctx.info = plan, info
        return params[0].new_zeros(token_size(plan))

    @staticmethod
    def backward(ctx, d_token):
        plan, info = ctx.plan, ctx.info
        per_head = token_size(plan) // plan.K
        grads = []
        for k, spec in enumerate(plan.heads):
            n_params = len(head_parameters(spec))
            if d_token is None or not (info["used"] >> k) & 1:
                grads += [None] * n_params
                continue
            L, sd = _layers(spec), spec.sd
            part = d_token[k * per_head:(k + 1) * per_head]
            o = 0
            dW = part[o:o + L * U * U].view(L, U, U); o += L * U * U
            db = part[o:o + (L + 1) * U].view(L + 1, U); o += (L + 1) * U
            g_in = part[o:o + U * sd].view(U, sd); o += U * sd
            g_out = part[o:o + U]; o += U
            g, _ = _grads_for_head(spec, dW, db, g_in, g_out, part[o:o + 1])
            grads += g
        return (None, None, *grads)


def _layers(spec) -> int:
    return 2 * len(spec.state[1]) + 1 + 2 * len(spec.shared[1])


def token_size(plan) -> int:
    spec = plan.heads[0]
    L, sd = _layers(spec), spec.sd
    return plan.K * (L * U * U + (L + 1) * U + U * sd + U + 1)


class FusedHeads(torch.autograd.Function):
    """(states, eps, dynamics row, head rows, gradient token of the head parameters) -> (moved, ll[K, N, M])."""

    @staticmethod
    def forward(ctx, plan, states, eps, dyn_row, head_rows, enabled_mask, precision, token, info):
        info["used"] |= enabled_mask
        N, M, sd = states.shape
        dev = states.device
        plan.refresh(dev, backward=True)
        rowbias = torch.cat([dyn_row[None], head_rows.detach()]).contiguous()
        moved, ll, act = ops.pf_heads_forward_train(plan.struct, states.detach(), eps, rowbias, enabled_mask,
                                                    precision=precision)
        if enabled_mask != (1 << plan.K) - 1:
            # planes of disabled heads are never written by the kernel: clear them here, once, so that backward can
            # treat the saved tensor as read-only (retain_graph / a second backward see the same values)
            for k in range(plan.K):
                if not (enabled_mask >> k) & 1:
                    act[k].zero_()
        ctx.plan, ctx.mask, ctx.shape = plan, enabled_mask, (N, M, sd)
        ctx.save_for_backward(act, moved)
        ctx.mark_non_differentiable(moved)
        return moved, ll

    @staticmethod
    def backward(ctx, _d_moved, d_ll):
        plan, mask = ctx.plan, ctx.mask
        N, M, sd = ctx.shape
        act, moved = ctx.saved_tensors
        d_ll = torch.nan_to_num(d_ll.contiguous(), nan=0.0)
        delta = ops.pf_heads_backward(plan.struct, N, M, act, d_ll, mask)
        if mask != (1 << plan.K) - 1:  # planes of disabled heads are never written by the kernels
            for k in range(plan.K):
                if not (mask >> k) & 1:
                    delta[k].zero_()
        moved_flat = moved.reshape(N * M, sd)
        dW, db, g_in, g_out = ops.pf_heads_weight_grads(act, delta, moved_flat, d_ll.reshape(plan.K, N * M))
        K = plan.K
        # per-trajectory row gradients: the mid layer's delta summed over the particles (chunk-major planes -> (N, 64))
        mid_layer = mid_layer_index(plan.heads[0])
        d_rows = delta[:, mid_layer].view(K, U // 4, N, M, 4).sum(dim=3).permute(0, 2, 1, 3).reshape(K, N, U)
        # this step's parameter gradients as ONE flat tensor, per head [dW | db | g_in | g_out | sum d_ll] (HeadGradToken)
        d_token = torch.cat([dW.reshape(K, -1), db.reshape(K, -1), g_in.reshape(K, -1), g_out.reshape(K, -1),
                             d_ll.reshape(K, -1).sum(dim=1, keepdim=True)], dim=1).reshape(-1)
        return (None, None, None, None, d_rows, None, None, d_token, None)


class Reweight(torch.autograd.Function):
    """(ll[K, N, M], modality log-weights (N, K) | None, logw_in (N, M), moved states) -> (normalised logw (N, M), estimate
    (N, sd)): fusion over the enabled heads, reweighting, normalisation and the weighted-average estimate of A.3 in one
    kernel, and their reverse mode in one more (``mmf_pf_reweight_train_fwd / _bwd``; the backward recomputes instead of
    saving intermediates).  The particle states carry no gradient (frozen dynamics)."""

    @staticmethod
    def forward(ctx, ll, modw, logw_in, states, enabled_mask):
        ll, logw_in, states = ll.contiguous(), logw_in.contiguous(), states.detach().contiguous()
        modw = None if modw is None else modw.contiguous()
        logw, est = ops.pf_reweight_train_fwd(ll.detach(), None if modw is None else modw.detach(), logw_in.detach(), states,
                                              enabled_mask)
        ctx.mask = enabled_mask
        ctx.has_modw = modw is not None
        ctx.save_for_backward(ll, logw_in, states, *([modw] if modw is not None else []))
        ctx.set_materialize_grads(False)
        return logw, est

    @staticmethod
    def backward(ctx, d_logw, d_est):
        ll, logw_in, states, *rest = ctx.saved_tensors
        modw = rest[0] if ctx.has_modw else None
        d_ll, d_w, d_in = ops.pf_reweight_train_bwd(ll, modw, logw_in, states, ctx.mask, d_est, d_logw)
        return d_ll, d_w, d_in, None, None


class FusedEKFLoop(torch.autograd.Function):
    """(plan, mean0 (F,N,sd), cov0 (F,N,sd,sd), controls (T,N,cd), z (F,T,N,sd), r_tril (F,T,N,sd,sd)) -> (means
    (F,T,N,sd), covs (F,T,N,sd,sd)): F extended Kalman filters over T steps in one launch (``mmf_ekf_loop_train_fwd``),
    and the reverse mode in one more (``mmf_ekf_loop_bwd``), which returns the gradients of mean0, cov0, z and r_tril.

    The dynamics are frozen and the reference evaluates their Jacobian A at a detached state (A.4), so A carries no
    gradient and the backward is SD x SD algebra given A and mu- of every step: the forward records both (the tape)
    instead of the backward re-running the dynamics MLP.  The controls receive no gradient (the dynamics are frozen
    and the controls are data)."""

    @staticmethod
    def forward(ctx, plan, mean0, cov0, controls, z, r_tril):
        cov0, z, r_tril = cov0.detach().contiguous(), z.detach().contiguous(), r_tril.detach().contiguous()
        means, covs, pred, jac = plan.loop_train(mean0.detach().contiguous(), cov0, controls.detach(), z, r_tril)
        # the structs (q_tril) and the weight buffers they point at, as of this forward
        ctx.structs, ctx.buffers = plan.structs, plan._buffers
        ctx.save_for_backward(cov0, z, r_tril, covs, pred, jac)
        ctx.set_materialize_grads(False)
        return means, covs

    @staticmethod
    def backward(ctx, d_means, d_covs):
        if d_means is None and d_covs is None:
            return None, None, None, None, None, None
        cov0, z, r_tril, covs, pred, jac = ctx.saved_tensors
        d_mean0, d_cov0, d_z, d_r = ops.ekf_loop_bwd(ctx.structs, cov0, z, r_tril, covs, pred, jac, d_means, d_covs)
        return None, d_mean0, d_cov0, None, d_z, d_r


def ekf_train_structure_ok(owner, filters, plan) -> bool:
    """The checks of ``fused_ekf_train_applicable`` that need no device: a recognised plan, ``owner.fused_train``, no
    hooks anywhere in ``owner`` (the fused step never calls the dynamics modules) and frozen dynamics in every filter
    (gradients into the dynamics MLP are not part of the kernels' adjoint)."""
    if plan is None or not getattr(owner, "fused_train", True):
        return False
    if any(m._forward_hooks or m._forward_pre_hooks for m in owner.modules()):
        return False
    return not any(p.requires_grad for f in filters for p in f.dynamics_model.parameters())


def fused_ekf_train_applicable(owner, filters, plan, controls, observations, beliefs) -> bool:
    """Train the EKF recursion of ``filters`` (the enabled filters of ``owner``) through ``FusedEKFLoop``: a gradient
    is needed (grad mode on, and a parameter of ``owner`` or one of the ``beliefs`` requires it), the structural checks
    of ``ekf_train_structure_ok`` pass, and controls and observations are CUDA fp32 tensors."""
    if not torch.is_grad_enabled():
        return False
    if not (any(t is not None and t.requires_grad for t in beliefs) or any(p.requires_grad for p in owner.parameters())):
        return False
    if not ekf_train_structure_ok(owner, filters, plan):
        return False
    tensors = [controls, *(observations.values() if isinstance(observations, dict) else [observations])]
    return all(isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 for t in tensors)


def fused_train_applicable(filt, plan, resample: bool) -> bool:
    """The fused training step covers exactly the reference's setting: no resampling, frozen dynamics,
    particle states without gradient, tensor-core precision."""
    if plan is None or resample or filt.precision not in ("bf16x3", "bf16"):
        return False
    if filt.particle_states.requires_grad:
        return False
    return not any(p.requires_grad for p in filt.dynamics_model.parameters())
