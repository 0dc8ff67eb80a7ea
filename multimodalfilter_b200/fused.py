"""Host-side "plans": recognise the reference's architectures inside a filter object, pack their
weights into the layouts ``include/mmf_b200.h`` documents, and drive the CUDA kernels.

Recognition is structural + by class name, NOT by ``isinstance`` on this package's classes, so the
reference's own ``crossmodal.push_models.PushCrossmodalParticleFilter`` (running on top of this
package's ``torchfilter`` drop-in) takes the fused path too.  A model that does not match keeps
working through the generic path of ``torchfilter.filters`` (user modules run as torch modules on
the GPU; the reweight / normalise / resample stages still run in the CUDA kernels).
"""
import math
from typing import List, Optional

import torch
import torch.nn as nn

from . import _lib, ops

U = _lib.UNITS

FUSABLE_DYNAMICS = {"PushDynamicsModel", "DoorDynamicsModel", "DoorDynamicsModelBrent"}
FUSABLE_HEADS = {"PushMeasurementModel", "DoorMeasurementModel"}
OBS_ORDER = (("image", "observation_image_layers"), ("pos", "observation_pos_layers"), ("sensors", "observation_sensors_layers"))
OBS_KEY = {"image": "image", "pos": "gripper_pos", "sensors": "gripper_sensors"}


# ------------------------------------------------------------------------------------------------
# structure parsing
# ------------------------------------------------------------------------------------------------
def _is_resblock(m) -> bool:
    b1, b2 = getattr(m, "block1", None), getattr(m, "block2", None)
    if not (isinstance(b1, nn.Linear) and isinstance(b2, nn.Linear)):
        return False
    act = getattr(m, "activation", None)
    if act is not None and not isinstance(act, nn.ReLU):
        return False
    return b1.in_features == U and b1.out_features == U and b2.in_features == U and b2.out_features == U


def _tokens(seq: nn.Sequential):
    out = []
    for m in seq:
        if isinstance(m, nn.Linear):
            out.append(("lin", m))
        elif isinstance(m, nn.ReLU):
            out.append(("relu", None))
        elif _is_resblock(m):
            out.append(("res", m))
        else:
            return None
    return out


def _parse_encoder(seq):
    """Linear(in, 64) -> ReLU -> resblock(64)   (ref: crossmodal/push_models/layers.py:20-24)."""
    t = _tokens(seq) if isinstance(seq, nn.Sequential) else None
    if not t or [k for k, _ in t] != ["lin", "relu", "res"] or t[0][1].out_features != U:
        return None
    return t[0][1], [t[2][1]]


def _parse_shared(seq, mid_relu: bool, out_dim: int):
    """Linear(64*k, 64) [-> ReLU] -> resblock* -> Linear(64, out_dim)."""
    t = _tokens(seq) if isinstance(seq, nn.Sequential) else None
    if not t or t[0][0] != "lin" or t[-1][0] != "lin":
        return None
    body = t[1:-1]
    if mid_relu:
        if not body or body[0][0] != "relu":
            return None
        body = body[1:]
    if any(k != "res" for k, _ in body):
        return None
    mid, out = t[0][1], t[-1][1]
    if mid.out_features != U or out.in_features != U or out.out_features != out_dim:
        return None
    return mid, [m for _, m in body], out


# ------------------------------------------------------------------------------------------------
# packing (layouts: include/mmf_b200.h, mmf_chain / mmf_traj_rows)
# ------------------------------------------------------------------------------------------------
def _t(w):  # (out, in) -> input-major (in, out), flattened
    return w.detach().t().contiguous().reshape(-1)


def _res_parts(blocks):
    parts = []
    for r in blocks:
        parts += [_t(r.block1.weight), r.block1.bias.detach(), _t(r.block2.weight), r.block2.bias.detach()]
    return parts


def pack_chain(in_lin, pre_res, mid_lin, state_cols: slice, post_res, out_lin) -> torch.Tensor:
    parts = [_t(in_lin.weight), in_lin.bias.detach()]
    parts += _res_parts(pre_res)
    parts.append(_t(mid_lin.weight[:, state_cols]))
    parts += _res_parts(post_res)
    parts += [out_lin.weight.detach().contiguous().reshape(-1), out_lin.bias.detach()]
    return torch.cat([p.reshape(-1).float() for p in parts]).contiguous()


def pack_rows(encoder, mid_lin, traj_cols: slice) -> torch.Tensor:
    parts = []
    if encoder is not None:
        enc_lin, enc_res = encoder
        parts += [_t(enc_lin.weight), enc_lin.bias.detach()] + _res_parts(enc_res)
    parts += [_t(mid_lin.weight[:, traj_cols]), mid_lin.bias.detach()]
    return torch.cat([p.reshape(-1).float() for p in parts]).contiguous()


def _chain_struct(w, in_dim, n_pre, mid_relu, n_post, out_dim):
    c = _lib.Chain()
    c.in_dim, c.n_pre_res, c.mid_relu, c.n_post_res, c.out_dim = in_dim, n_pre, int(mid_relu), n_post, out_dim
    c.w = w.data_ptr()
    c.w_mma = None
    return c


def _rows_struct(w, in_dim, has_encoder):
    r = _lib.TrajRows()
    r.in_dim, r.has_encoder, r.w = in_dim, int(has_encoder), w.data_ptr()
    return r


def _q_tril(dyn, sd):
    if hasattr(dyn, "Q_scale_tril_diag"):
        return torch.diag(dyn.Q_scale_tril_diag.detach()).float().cpu()
    return dyn.Q_scale_tril.detach().float().cpu()


class _DynamicsSpec:
    """Parsed gated-residual dynamics (ref: crossmodal/push_models/dynamics.py:10-64)."""

    def __init__(self, dyn):
        self.ok = False
        if type(dyn).__name__ not in FUSABLE_DYNAMICS and not getattr(dyn, "_mmf_fusable", False):
            return
        sd = dyn.state_dim
        st = _parse_encoder(getattr(dyn, "state_layers", None))
        ct = _parse_encoder(getattr(dyn, "control_layers", None))
        sh = _parse_shared(getattr(dyn, "shared_layers", None), mid_relu=False, out_dim=sd + 1)
        if not (st and ct and sh) or st[0].in_features != sd or sh[0].in_features != 2 * U:
            return
        if not (hasattr(dyn, "Q_scale_tril") or hasattr(dyn, "Q_scale_tril_diag")):
            return
        self.dyn, self.sd, self.cd = dyn, sd, ct[0].in_features
        self.state, self.control, self.shared = st, ct, sh
        self.ok = 1 <= sd <= _lib.MAX_SD and 1 <= self.cd <= _lib.MAX_CD

    def pack(self):
        (in_lin, pre), (mid, post, out) = self.state, self.shared
        # cat order is (control_features, state_features): ref: dynamics.py:50
        chain = pack_chain(in_lin, pre, mid, slice(U, 2 * U), post, out)
        rows = pack_rows(self.control, mid, slice(0, U))
        return chain, rows

    def structs(self, chain, rows):
        (_, pre), (_, post, _) = self.state, self.shared
        c = _chain_struct(chain, self.sd, len(pre), False, len(post), self.sd + 1)
        r = _rows_struct(rows, self.cd, True)
        return c, r

    def q(self):
        q = torch.zeros(_lib.MAX_SD * _lib.MAX_SD)
        q[: self.sd * self.sd] = _q_tril(self.dyn, self.sd).reshape(-1)
        return q

    def parameters(self):
        return list(self.dyn.parameters())


class _HeadSpec:
    """Parsed per-particle measurement head (ref: crossmodal/push_models/pf.py:30-109)."""

    def __init__(self, head, sd):
        self.ok = False
        if type(head).__name__ not in FUSABLE_HEADS and not getattr(head, "_mmf_fusable", False):
            return
        mods = getattr(head, "modalities", None)
        st = _parse_encoder(getattr(head, "state_layers", None))
        sh = _parse_shared(getattr(head, "shared_layers", None), mid_relu=True, out_dim=1)
        if not (mods and st and sh) or st[0].in_features != sd:
            return
        self.head = head
        self.encoders = [(OBS_KEY[m], getattr(head, attr)) for m, attr in OBS_ORDER if m in mods]
        self.feat_dim = U * len(self.encoders)
        if sh[0].in_features != self.feat_dim + U or self.feat_dim > 256:
            return
        self.sd, self.state, self.shared = sd, st, sh
        self.ok = True

    def pack(self):
        (in_lin, pre), (mid, post, out) = self.state, self.shared
        # cat order is (observation_features, state_features): ref: pf.py:101
        chain = pack_chain(in_lin, pre, mid, slice(self.feat_dim, self.feat_dim + U), post, out)
        rows = pack_rows(None, mid, slice(0, self.feat_dim))
        return chain, rows

    def structs(self, chain, rows):
        (_, pre), (_, post, _) = self.state, self.shared
        return _chain_struct(chain, self.sd, len(pre), True, len(post), 1), _rows_struct(rows, self.feat_dim, False)

    def _feature_program(self):
        """Encoders of the non-image modalities + the concatenation as one mmf_row_mlp launch; the image features
        (CNN trunk kernel + Linear tail) enter as an input."""
        prog = RowProgram()
        base = prog.alloc(self.feat_dim, fresh=True)
        for i, (key, enc) in enumerate(self.encoders):
            if key == "image":
                prog.input(U, slot=base + U * i)
            else:
                src = prog.input(enc[0].in_features)
                prog.sequential(enc, src, enc[0].in_features, dst=base + U * i)
                prog.release(src, enc[0].in_features)
        prog.output(base, self.feat_dim)
        return prog

    def observation_features(self, observations) -> torch.Tensor:
        """(B, feat_dim) for a dict of (B, ...) observations (ref: pf.py:76-88, order image/pos/sensors)."""
        raw = [observations[key] for key, _ in self.encoders if key != "image"]
        if raw and row_program_ok(*raw):
            prog = cached_program(self.head, "features", self._feature_program)
            if prog is not None:
                ins = []
                for key, enc in self.encoders:
                    x = observations[key]
                    ins.append(enc(x[:, None, :, :]) if key == "image" else x)
                return prog.run(ins)[0]
        feats = []
        for key, enc in self.encoders:
            x = observations[key]
            feats.append(enc(x[:, None, :, :] if key == "image" else x))
        return torch.cat(feats, dim=1) if len(feats) > 1 else feats[0]


def _versions(params):
    return tuple((p.data_ptr(), p._version) for p in params)


class PFPlan:
    """Fused particle-filter step for a recognised (dynamics, measurement) pair."""

    def __init__(self, dyn_spec, head_specs, measurement_model, composite: bool):
        self.dyn = dyn_spec
        self.heads: List[_HeadSpec] = head_specs
        self.mm = measurement_model
        self.composite = composite  # CrossmodalParticleFilterMeasurementModel vs a single head
        self.K = len(head_specs)
        self.sd, self.cd = dyn_spec.sd, dyn_spec.cd
        self._sig = None
        self._buffers = None
        self._has_bwd = False
        self.struct = None

    @staticmethod
    def build(filt) -> Optional["PFPlan"]:
        dyn = _DynamicsSpec(filt.dynamics_model)
        if not dyn.ok:
            return None
        mm = filt.measurement_model
        if hasattr(mm, "measurement_models") and hasattr(mm, "_enabled_models"):
            if type(mm).__name__ != "CrossmodalParticleFilterMeasurementModel" and not getattr(mm, "_mmf_fusable", False):
                return None
            heads = [_HeadSpec(h, dyn.sd) for h in mm.measurement_models]
            composite = True
        else:
            heads = [_HeadSpec(mm, dyn.sd)]
            composite = False
        if not heads or len(heads) > _lib.MAX_HEADS or not all(h.ok for h in heads):
            return None
        return PFPlan(dyn, heads, mm, composite)

    # -- weights ------------------------------------------------------------------------------------
    def _params(self):
        ps = self.dyn.parameters()
        for h in self.heads:
            ps += list(h.head.state_layers.parameters()) + list(h.head.shared_layers.parameters())
        return ps

    def refresh(self, device, backward: bool = False):
        params = self._params()
        sig = (str(device), _versions(params))
        if sig == self._sig and (not backward or self._has_bwd):
            return
        if any(p.device != device for p in params):
            raise _lib.MMFError("filter parameters must live on the CUDA device of the inputs (call .to(device))")
        bufs = []
        m = _lib.PFModel()
        m.state_dim, m.control_dim, m.num_heads = self.sd, self.cd, self.K
        chain, rows = self.dyn.pack()
        bufs += [chain, rows]
        m.dynamics, m.dynamics_rows = self.dyn.structs(chain, rows)
        for k, h in enumerate(self.heads):
            chain, rows = h.pack()
            bufs += [chain, rows]
            m.heads[k], m.head_rows[k] = h.structs(chain, rows)
        q = self.dyn.q()
        for i in range(_lib.MAX_SD * _lib.MAX_SD):
            m.q_tril[i] = float(q[i])
        # tcgen05 operand images (bf16 hi/lo halves in the UMMA shared-memory layout)
        bufs.append(ops.pack_chain_mma(m.dynamics, device))
        for k in range(self.K):
            bufs.append(ops.pack_chain_mma(m.heads[k], device))
            if backward:
                bufs.append(ops.pack_chain_bwd(m.heads[k], device))
        self._has_bwd = backward
        self._buffers, self.struct, self._sig = bufs, m, sig

    # -- per-trajectory inputs ------------------------------------------------------------------------
    def enabled(self) -> List[bool]:
        return list(self.mm._enabled_models) if self.composite else [True]

    def enabled_mask(self) -> int:
        return sum(1 << k for k, on in enumerate(self.enabled()) if on)

    def head_features(self, observations) -> List[Optional[torch.Tensor]]:
        """Observation features of every enabled head for a flat batch of observations."""
        return [h.observation_features(observations) if on else None for h, on in zip(self.heads, self.enabled())]

    def modality_log_weights(self, observations) -> Optional[torch.Tensor]:
        """(B, K) raw log-weights over ALL heads, or None for the un-weighted fusion
        (ref: crossmodal/base_models/crossmodal_pf.py:116-121,136-139)."""
        wm = getattr(self.mm, "crossmodal_weight_model", None) if self.composite else None
        if wm is None:
            return None
        w = wm(observations=observations)
        assert w.shape[1] == self.K, f"weight model returned {tuple(w.shape)}, expected (N, {self.K})"
        return w

    # -- one step ---------------------------------------------------------------------------------------
    def step(self, states, logw, controls, feats, modw, eps, *, precision, estimation, mode, alpha, M_out, uniforms,
             want_debug=False):
        self.refresh(states.device)
        N = states.shape[0]
        # upstream asserts len(controls) == N; here a mismatch would make the kernels index rows out of bounds
        assert controls.shape[0] == N, f"controls have {controls.shape[0]} rows for {N} trajectories"
        assert len(feats) == self.K and all(f is None or f.shape[0] == N for f in feats), "observation features / N mismatch"
        assert modw is None or modw.shape[0] == N, "modality weights / N mismatch"
        rowbias = ops.pf_traj_rows(self.struct, self.K, controls, feats)
        res = ops.pf_predict_measure(self.struct, states, eps, rowbias, logw, modw, self.enabled_mask(),
                                     precision=precision, want_ll=want_debug)
        moved, logw_unnorm = res[0], res[1]
        out = ops.pf_normalize_resample(moved, logw_unnorm, estimation=estimation, mode=mode, alpha=alpha,
                                        M_out=M_out, uniforms=uniforms, want_debug=want_debug)
        if want_debug:
            out.update(moved=moved, logw_unnorm=logw_unnorm, ll=res[2], rowbias=rowbias)
        return out


class EKFPlan:
    """Fused EKF recursion for VirtualSensorExtendedKalmanFilter(s) with recognised dynamics."""

    def __init__(self, dyn_specs):
        self.dyns = dyn_specs
        self.sd, self.cd = dyn_specs[0].sd, dyn_specs[0].cd
        self._sig = None
        self._buffers = None
        self.structs = None

    @staticmethod
    def build(filters) -> Optional["EKFPlan"]:
        specs = [_DynamicsSpec(f.dynamics_model) for f in filters]
        if not specs or len(specs) > 4 or not all(s.ok for s in specs):
            return None
        if any(s.sd != specs[0].sd or s.cd != specs[0].cd for s in specs):
            return None
        return EKFPlan(specs)

    def refresh(self, device):
        params = [p for s in self.dyns for p in s.parameters()]
        sig = (str(device), _versions(params))
        if sig == self._sig:
            return
        if any(p.device != device for p in params):
            raise _lib.MMFError("filter parameters must live on the CUDA device of the inputs (call .to(device))")
        bufs, structs = [], []
        for s in self.dyns:
            chain, rows = s.pack()
            bufs += [chain, rows]
            m = _lib.EKFModel()
            m.state_dim, m.control_dim = s.sd, s.cd
            m.dynamics, m.dynamics_rows = s.structs(chain, rows)
            q = s.q()
            for i in range(_lib.MAX_SD * _lib.MAX_SD):
                m.q_tril[i] = float(q[i])
            structs.append(m)
        self._buffers, self.structs, self._sig = bufs, structs, sig

    def loop(self, mean0, cov0, controls, z, r_tril):
        """mean0 (F,N,sd), cov0 (F,N,sd,sd), controls (T,N,cd), z (F,T,N,sd), r_tril (F,T,N,sd,sd)."""
        self.refresh(z.device)
        return ops.ekf_loop(self.structs, mean0, cov0, controls, z, r_tril)

    def loop_train(self, mean0, cov0, controls, z, r_tril):
        """``loop`` plus the tape of the backward: -> means, covs, pred (F,T,N,sd), jac (F,T,N,sd,sd)."""
        self.refresh(z.device)
        return ops.ekf_loop_train(self.structs, mean0, cov0, controls, z, r_tril)

    def jacobian(self, which, states, controls):
        self.refresh(states.device)
        return ops.dynamics_jacobian(self.structs[which], states, controls)


# ------------------------------------------------------------------------------------------------
# per-trajectory MLP stacks -> one-launch programs (mmf_row_mlp)
# ------------------------------------------------------------------------------------------------
class NotFusable(Exception):
    pass


class RowProgram:
    """A stack of Linear / ReLU / Sigmoid / fannypack resblocks over per-trajectory rows, compiled for ``mmf_row_mlp``:
    a list of fused ops ``dst = act(W src + b [+ res])`` over scratch slots (float offsets into a per-row scratch),
    the input-major weight pack, and the input / output slots.  Build with ``input`` / ``sequential`` / ``output``;
    ``run`` repacks the weights when a parameter changed."""

    def __init__(self):
        self.ops, self.params, self._w_floats, self.scratch = [], [], 0, 0
        self.in_slots, self.in_dims, self.out_slots, self.out_dims = [], [], [], []
        self._packed = None
        self._free = []  # (slot, size) of dead temporaries: the per-row scratch lives in shared memory, so it is reused

    def alloc(self, dim: int, fresh: bool = False) -> int:
        """A scratch slot; ``fresh`` = never a recycled one (program inputs: they are all written before the first op runs)."""
        size = ((dim + 3) // 4) * 4
        fits = [] if fresh else [f for f in self._free if f[1] >= size]
        if fits:
            slot, have = min(fits, key=lambda f: f[1])
            self._free.remove((slot, have))
            if have > size:
                self._free.append((slot + size, have - size))
            return slot
        slot, self.scratch = self.scratch, self.scratch + size
        return slot

    def release(self, slot: int, dim: int) -> None:
        """A temporary nobody reads any more (the kernel requires dst to differ from src / res of the SAME op only)."""
        self._free.append((slot, ((dim + 3) // 4) * 4))
        merged = []
        for start, size in sorted(self._free):  # coalesce neighbours: two dead 64-wide slots hold a 128-wide layer
            if merged and merged[-1][0] + merged[-1][1] == start:
                merged[-1] = (merged[-1][0], merged[-1][1] + size)
            else:
                merged.append((start, size))
        self._free = merged

    def input(self, dim: int, slot: int = None) -> int:
        slot = self.alloc(dim, fresh=True) if slot is None else slot
        self.in_slots.append(slot)
        self.in_dims.append(dim)
        return slot

    def output(self, slot: int, dim: int) -> None:
        self.out_slots.append(slot)
        self.out_dims.append(dim)

    def _linear(self, lin: nn.Linear, src: int, act: int, res: int = -1, dst: int = None) -> int:
        if lin.bias is None or lin.out_features > 256:
            raise NotFusable("Linear without bias or wider than 256")
        dst = self.alloc(lin.out_features) if dst is None else dst
        op = _lib.MlpOp()
        op.in_dim, op.out_dim, op.act, op.src, op.dst, op.res, op.w_off = (
            lin.in_features, lin.out_features, act, src, dst, res, self._w_floats)
        self.ops.append(op)
        self.params.append(lin)
        self._w_floats += lin.in_features * lin.out_features + lin.out_features
        if len(self.ops) > _lib.MLP_MAX_OPS:
            raise NotFusable("program too long")
        return dst

    def sequential(self, seq, src: int, src_dim: int, dst: int = None):
        """Append the modules of an nn.Sequential (or a list); the LAST op writes to ``dst`` when given.
        Returns (slot, dim) of the result."""
        mods = list(seq)
        cur, dim, i = src, src_dim, 0
        mine = set()  # temporaries this call allocated: dead once the next op has consumed them

        def advance(new, new_dim, *dead):
            for slot, d in dead:
                if slot in mine:
                    mine.discard(slot)
                    self.release(slot, d)
            if dst is None or new != dst:
                mine.add(new)
            return new, new_dim

        while i < len(mods):
            m = mods[i]
            last = lambda consumed: i + consumed >= len(mods)  # noqa: E731
            if isinstance(m, nn.Linear):
                if m.in_features != dim:
                    raise NotFusable("width mismatch")
                act, used = _lib.MLP_NONE, 1
                if i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU):
                    act, used = _lib.MLP_RELU, 2
                elif i + 1 < len(mods) and isinstance(mods[i + 1], nn.Sigmoid):
                    act, used = _lib.MLP_SIGMOID, 2
                new = self._linear(m, cur, act, dst=dst if last(used) else None)
                cur, dim = advance(new, m.out_features, (cur, dim))
                i += used
            elif isinstance(getattr(m, "block1", None), nn.Linear) and isinstance(getattr(m, "block2", None), nn.Linear):
                act = getattr(m, "activation", None)
                if (act is not None and not isinstance(act, nn.ReLU)) or m.block1.in_features != dim \
                        or m.block2.out_features != dim or m.block1.out_features != m.block2.in_features:
                    raise NotFusable("unsupported residual block")
                t = self._linear(m.block1, cur, _lib.MLP_RELU)
                mine.add(t)
                new = self._linear(m.block2, t, _lib.MLP_RELU, res=cur, dst=dst if last(1) else None)
                cur, dim = advance(new, dim, (t, m.block1.out_features), (cur, dim))
                i += 1
            else:
                raise NotFusable(f"unsupported module {type(m).__name__}")
        mine.discard(cur)  # the result stays live: it belongs to the caller
        return cur, dim

    def _weights(self, device):
        sig = (str(device), tuple((p.data_ptr(), p._version) for lin in self.params for p in (lin.weight, lin.bias)))
        if self._packed is None or self._packed[0] != sig:
            parts = []
            for lin in self.params:
                parts += [lin.weight.detach().t().contiguous().reshape(-1), lin.bias.detach().reshape(-1)]
            self._packed = (sig, torch.cat([p.float() for p in parts]).to(device).contiguous())
        return self._packed[1]

    def run(self, inputs):
        assert len(inputs) == len(self.in_slots) and all(x.shape[1] == d for x, d in zip(inputs, self.in_dims))
        return ops.row_mlp(self.ops, self._weights(inputs[0].device), inputs, self.in_slots, self.out_dims, self.out_slots,
                           self.scratch)


def row_program_ok(*tensors) -> bool:
    """The one-launch programs serve inference on CUDA fp32 rows; anything else keeps the torch modules."""
    return not torch.is_grad_enabled() and all(t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 for t in tensors)


def cached_program(owner, key, build):
    """Per-module cache of compiled programs (None = the stack is not fusable: keep the torch path)."""
    cache = owner.__dict__.setdefault("_mmf_programs", {})
    if key not in cache:
        try:
            cache[key] = build()
        except NotFusable:
            cache[key] = None
    return cache[key]


def flatten_time(observations, T, N):
    """dict of (T, N, ...) -> dict of (T*N, ...)."""
    return {k: v.reshape(T * N, *v.shape[2:]) for k, v in observations.items()}


class StagedObservations(dict):
    """Observation dict whose (T, N, ...) tensors are being copied host -> device, chunk by chunk over the flattened
    T*N rows, on a side stream.  ``ready(hi)`` makes the current stream wait until rows [0, hi) have landed, so the
    encoders of chunk c run while chunk c+1 is still on the PCIe bus (end-to-end ``forward_loop`` from pinned host
    buffers: the copy disappears behind the encoder kernels)."""

    def __init__(self, host_observations, device, T, N, chunk_rows):
        super().__init__()
        self.chunk_rows = chunk_rows
        self.events = []
        total = T * N
        side = torch.cuda.Stream(device=device)
        flat_src = {}
        for k, v in host_observations.items():
            self[k] = torch.empty(v.shape, dtype=v.dtype, device=device)
            flat_src[k] = v.reshape(total, *v.shape[2:])
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            for lo in range(0, total, chunk_rows):
                hi = min(total, lo + chunk_rows)
                for k, dst in self.items():
                    dst.reshape(total, *dst.shape[2:])[lo:hi].copy_(flat_src[k][lo:hi], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(side)
                self.events.append(ev)
        for dst in self.values():
            dst.record_stream(side)

    def ready(self, hi):
        torch.cuda.current_stream().wait_event(self.events[(hi + self.chunk_rows - 1) // self.chunk_rows - 1])


def batched_over_time(fn, observations, T, N, chunk_rows=16384):
    """Run a per-trajectory module once over all T*N rows (chunked to bound CNN activations)."""
    flat = flatten_time(observations, T, N)
    total = T * N
    staged = isinstance(observations, StagedObservations)
    if staged:
        chunk_rows = observations.chunk_rows
    outs = []
    for lo in range(0, total, chunk_rows):
        hi = min(total, lo + chunk_rows)
        if staged:
            observations.ready(hi)
        outs.append(fn({k: v[lo:hi] for k, v in flat.items()}))
    return outs


def log_num(M: int) -> float:
    return -math.log(M)
